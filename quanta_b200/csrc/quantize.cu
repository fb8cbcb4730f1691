// Quantize kernels (rows A1-A3, B1 of SURVEY §8) and their C-ABI entry points.
//
// Hot kernel: quantize_rows_tma_kernel — a persistent, warp-specialised stream:
//   * one producer warp feeds a 3-stage shared-memory ring with 32 KB TMA tiles
//     (cp.async.bulk.tensor, 256 rows x 128 B, SWIZZLE_128B, L2 evict-first),
//   * 256 consumer threads each own one 32-element row: the swizzle makes the
//     8 x LDS.128 of a row bank-conflict free and leaves the row in natural
//     order in registers, so a 64-element block is one shuffle away and the
//     packed codes leave as ONE aligned 128-bit store per thread.
// Arithmetic is bit-exact with the reference's eager torch chain (see
// common.cuh: affine_params / affine_quotient / code_bits).
#include "common.cuh"

#include <cstdio>

namespace quanta {

// --------------------------------------------------------------------------
// conventions
// --------------------------------------------------------------------------
enum Conv : int { kConvA = 0, kConvBSym = 1, kConvBAsym = 2 };

// Per-group parameters as the element loop needs them.
struct ElemParams {
    // conv A: a = mn, s = scale, r = rcp (0 -> slow divide)
    // conv B: s = scale (multiplier), a = zp
    float a, s, r;
};

template <int CONV, bool ASSUME_FAST = false>
__device__ __forceinline__ uint32_t elem_code_bits(float x, const ElemParams& p, float L, float Q) {
    if (CONV == kConvA) {
        AffineParams ap{p.a, p.s, p.r, ASSUME_FAST || p.r != 0.0f};
        return code_bits(affine_quotient(x, ap), L);
    } else if (CONV == kConvBSym) {
        // q = clamp(round(x*scale), -Q, Q) (+OFF added by the packer); NaN -> 0
        float t = __fmul_rn(x, p.s);
        float c = fminf(fmaxf(t, -Q), Q);
        c = (t != t) ? 0.0f : c;
        return __float_as_uint(__fadd_rn(c, kMagic));
    } else {
        float t = __fadd_rn(__fmul_rn(x, p.s), p.a);
        return code_bits(t, L);
    }
}

// Pack N code words (kMagicBits + code) into bytes / nibbles with a Horner
// chain of IMADs; the magic offsets add up to a compile-time constant.
template <int CONV, int BITS>
__device__ __forceinline__ uint32_t pack_bytes4(uint32_t u0, uint32_t u1, uint32_t u2, uint32_t u3) {
    constexpr uint32_t off = (CONV == kConvBSym) ? (BITS == 8 ? 128u : 8u) : 0u;
    constexpr uint32_t k = (kMagicBits - off) * 0x01010101u;
    uint32_t acc = u3;
    acc = acc * 256u + u2;
    acc = acc * 256u + u1;
    acc = acc * 256u + u0;
    return acc - k;
}
template <int CONV>
__device__ __forceinline__ uint32_t pack_nibbles8(const uint32_t* u) {
    constexpr uint32_t off = (CONV == kConvBSym) ? 8u : 0u;
    constexpr uint32_t k = (kMagicBits - off) * 0x11111111u;
    uint32_t acc = u[7];
#pragma unroll
    for (int i = 6; i >= 0; --i) acc = acc * 16u + u[i];
    return acc - k;
}

// Parameters from (mn, mx) for the three conventions.  For conv B `close`
// returns torch.isclose(mn, mx) (backends/cpu/quantization.py:38).
__device__ __forceinline__ bool isclose_f32(float a, float b) {
    if (a == b) return true;
    float allowed = __fadd_rn(1e-8f, fabsf(__fmul_rn(1e-5f, b)));
    float actual = fabsf(__fsub_rn(a, b));
    return (fabsf(actual) <= 3.402823466e38f) && actual <= allowed;
}

template <int CONV>
__device__ __forceinline__ void group_params(float mn, float mx, int bits, float* scale, float* zp, float* rcp,
                                             bool* close) {
    const float L = bits == 8 ? 255.0f : 15.0f, Q = bits == 8 ? 127.0f : 7.0f;
    if (CONV == kConvA) {
        AffineParams p = affine_params(mn, mx, L);
        *scale = p.scale; *zp = p.mn; *rcp = p.rcp; *close = false;
    } else {
        *close = isclose_f32(mn, mx);
        if (CONV == kConvBSym) {
            float am = max_nan(fabsf(mn), fabsf(mx));
            *scale = __fmul_rn(__frcp_rn(am), Q);          // int / Tensor == reciprocal * int
            *zp = 0.0f;
        } else {
            float s = __fmul_rn(__frcp_rn(__fsub_rn(mx, mn)), L);
            *scale = s;
            *zp = rintf(__fmul_rn(-mn, s));
        }
        *rcp = 0.0f;
    }
}

// --------------------------------------------------------------------------
// workspace layout (floats): [0] early-out flag (int) | [64 ...] rcp per channel
// | partial min / max
// --------------------------------------------------------------------------
constexpr int kWsHeaderFloats = 64;
// one bit pattern from every 16-byte chunk of a loaded 32-element row (see mbar_arrive_after_loads)
template <typename T>
__device__ __forceinline__ uint32_t row_dep(const float* v) {
    constexpr int step = 16 / (int)sizeof(T);            // elements per chunk: 4 (fp32) or 8 (16-bit)
    uint32_t d = 0;
#pragma unroll
    for (int k = 0; k < 32; k += step) d ^= __float_as_uint(v[k]);
    return d;
}

constexpr int kMaxPartialCtas = kNumSMs * 8;
constexpr int kMaxDim0Chunks = 64;

// --------------------------------------------------------------------------
// 1. min/max reductions
// --------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) minmax_tensor_partial_kernel(const T* __restrict__ x, int64_t n,
                                                                    float* __restrict__ pmin,
                                                                    float* __restrict__ pmax) {
    pdl_wait();                                            // launched with programmatic stream serialization (launch_pdl)
    constexpr int VEC = 16 / sizeof(T);
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
    float mn = to_f32(x[0]), mx = mn;
    const bool aligned = (reinterpret_cast<uintptr_t>(x) & 15) == 0;
    int64_t nvec = aligned ? n / VEC : 0;
    const uint4* xv = reinterpret_cast<const uint4*>(x);
    int64_t i = tid;
    // 4 independent 128-bit loads in flight per thread
    for (; i + 3 * nthreads < nvec; i += 4 * nthreads) {
        uint4 v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = __ldg(xv + i + k * nthreads);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const T* e = reinterpret_cast<const T*>(&v[k]);
#pragma unroll
            for (int j = 0; j < VEC; ++j) { float f = to_f32(e[j]); mn = min_nan(mn, f); mx = max_nan(mx, f); }
        }
    }
    for (; i < nvec; i += nthreads) {
        uint4 v = __ldg(xv + i);
        const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
        for (int j = 0; j < VEC; ++j) { float f = to_f32(e[j]); mn = min_nan(mn, f); mx = max_nan(mx, f); }
    }
    for (int64_t j = nvec * VEC + tid; j < n; j += nthreads) {
        float f = to_f32(x[j]); mn = min_nan(mn, f); mx = max_nan(mx, f);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = min_nan(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    __shared__ float smn[8], smx[8];
    if ((threadIdx.x & 31) == 0) { smn[threadIdx.x >> 5] = mn; smx[threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) { mn = min_nan(mn, smn[w]); mx = max_nan(mx, smx[w]); }
        pmin[blockIdx.x] = mn; pmax[blockIdx.x] = mx;
    }
}

template <int CONV>
__global__ void __launch_bounds__(256) minmax_tensor_finalize_kernel(const float* __restrict__ pmin,
                                                                     const float* __restrict__ pmax, int nparts,
                                                                     int bits, float* scale_out, float* zp_out,
                                                                     float* ws) {
    pdl_wait();                                            // launched with programmatic stream serialization (launch_pdl)
    float mn = pmin[0], mx = pmax[0];
    for (int i = threadIdx.x; i < nparts; i += blockDim.x) { mn = min_nan(mn, pmin[i]); mx = max_nan(mx, pmax[i]); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = min_nan(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    __shared__ float smn[8], smx[8];
    if ((threadIdx.x & 31) == 0) { smn[threadIdx.x >> 5] = mn; smx[threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) { mn = min_nan(mn, smn[w]); mx = max_nan(mx, smx[w]); }
        float s, z, r; bool close;
        group_params<CONV>(mn, mx, bits, &s, &z, &r, &close);
        if (CONV != kConvA && close) { s = 1.0f; z = mn; }      // early-out: zeros, ones_like(min), min
        scale_out[0] = s; zp_out[0] = z;
        ws[kWsHeaderFloats] = r;
        reinterpret_cast<int*>(ws)[0] = (CONV != kConvA && close) ? 1 : 0;
    }
}

// dim 0: thread owns 4 consecutive columns, blockIdx.y owns a chunk of rows.
template <typename T>
__global__ void __launch_bounds__(128) minmax_dim0_partial_kernel(const T* __restrict__ x, int64_t rows, int64_t cols,
                                                                  int rows_per_chunk, float* __restrict__ pmin,
                                                                  float* __restrict__ pmax) {
    pdl_wait();                                            // launched with programmatic stream serialization (launch_pdl)
    const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (c >= cols) return;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r1 = min(rows, r0 + rows_per_chunk);
    float mn[4], mx[4];
    auto load4 = [&](int64_t r, float* f) {
        if (sizeof(T) == 4) {
            float4 v = __ldg(reinterpret_cast<const float4*>(x + r * cols + c));
            f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
        } else {
            uint2 v = __ldg(reinterpret_cast<const uint2*>(x + r * cols + c));
            const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
            for (int j = 0; j < 4; ++j) f[j] = to_f32(e[j]);
        }
    };
    load4(r0, mn);
#pragma unroll
    for (int j = 0; j < 4; ++j) mx[j] = mn[j];
    int64_t r = r0 + 1;
    for (; r + 3 < r1; r += 4) {
        float f[4][4];
#pragma unroll
        for (int k = 0; k < 4; ++k) load4(r + k, f[k]);
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int j = 0; j < 4; ++j) { mn[j] = min_nan(mn[j], f[k][j]); mx[j] = max_nan(mx[j], f[k][j]); }
    }
    for (; r < r1; ++r) {
        float f[4]; load4(r, f);
#pragma unroll
        for (int j = 0; j < 4; ++j) { mn[j] = min_nan(mn[j], f[j]); mx[j] = max_nan(mx[j], f[j]); }
    }
    float4* om = reinterpret_cast<float4*>(pmin + (int64_t)blockIdx.y * cols + c);
    float4* ox = reinterpret_cast<float4*>(pmax + (int64_t)blockIdx.y * cols + c);
    *om = make_float4(mn[0], mn[1], mn[2], mn[3]);
    *ox = make_float4(mx[0], mx[1], mx[2], mx[3]);
}

// generic dim-0 partial (any cols / alignment): one thread per column.
template <typename T>
__global__ void __launch_bounds__(128) minmax_dim0_partial_generic_kernel(const T* __restrict__ x, int64_t rows,
                                                                          int64_t cols, int rows_per_chunk,
                                                                          float* __restrict__ pmin,
                                                                          float* __restrict__ pmax) {
    pdl_wait();                                            // launched with programmatic stream serialization (launch_pdl)
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r1 = min(rows, r0 + rows_per_chunk);
    float mn = to_f32(x[r0 * cols + c]), mx = mn;
    for (int64_t r = r0 + 1; r < r1; ++r) { float f = to_f32(x[r * cols + c]); mn = min_nan(mn, f); mx = max_nan(mx, f); }
    pmin[(int64_t)blockIdx.y * cols + c] = mn;
    pmax[(int64_t)blockIdx.y * cols + c] = mx;
}

// Reduce the row-chunk partials of each column and emit its parameters; conv B
// also needs "allclose for ALL channels": every thread ANDs into ws[0]
// (pre-set to 1 by minmax_dim0_flag_init).
__global__ void dim0_flag_init_kernel(float* ws, int value) {
    pdl_wait();                                            // launched with programmatic stream serialization (launch_pdl)
    reinterpret_cast<int*>(ws)[0] = value;
}

template <int CONV>
__global__ void __launch_bounds__(32) minmax_dim0_finalize_kernel(const float* __restrict__ pmin,
                                                                   const float* __restrict__ pmax, int nchunks,
                                                                   int64_t cols, int bits, float* scale_out,
                                                                   float* zp_out, float* ws) {
    pdl_wait();                                            // launched with programmatic stream serialization (launch_pdl)
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool close = true;
    if (c < cols) {
        float mn = pmin[c], mx = pmax[c];
        int k = 1;
        for (; k + 7 < nchunks; k += 8) {                 // 16 independent loads in flight
            float a[8], b[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) { a[j] = pmin[(int64_t)(k + j) * cols + c]; b[j] = pmax[(int64_t)(k + j) * cols + c]; }
#pragma unroll
            for (int j = 0; j < 8; ++j) { mn = min_nan(mn, a[j]); mx = max_nan(mx, b[j]); }
        }
        for (; k < nchunks; ++k) { mn = min_nan(mn, pmin[(int64_t)k * cols + c]); mx = max_nan(mx, pmax[(int64_t)k * cols + c]); }
        float s, z, r;
        group_params<CONV>(mn, mx, bits, &s, &z, &r, &close);
        scale_out[c] = s; zp_out[c] = z;
        ws[kWsHeaderFloats + c] = (CONV == kConvA) ? r : mn;      // conv B keeps min for the early-out
    }
    if (CONV != kConvA) {
        int all = __syncthreads_and(close ? 1 : 0);
        if (threadIdx.x == 0 && !all) atomicAnd(reinterpret_cast<int*>(ws), 0);
    }
}

// conv B early-out for per_channel: scale = 1, zp = min for every channel.
__global__ void dim0_earlyout_params_kernel(int64_t cols, float* scale_out, float* zp_out, const float* ws) {
    pdl_wait();                                            // launched with programmatic stream serialization (launch_pdl)
    if (reinterpret_cast<const int*>(ws)[0] == 0) return;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < cols) { scale_out[c] = 1.0f; zp_out[c] = ws[kWsHeaderFloats + c]; }
}

// --------------------------------------------------------------------------
// 2. the streaming TMA kernel (BLOCK mode)
// --------------------------------------------------------------------------
constexpr int kRowElems = 32;          // elements owned by one consumer thread
constexpr int kTileRows = 256;         // rows (= consumer threads) per TMA tile
constexpr int kStages = 3;
constexpr int kConsumerWarps = kTileRows / 32;
constexpr int kTmaThreads = kTileRows + 32;

template <typename T> struct RowLayout {
    static constexpr int kRowBytes = kRowElems * sizeof(T);            // 128 (fp32) or 64 (16-bit)
    static constexpr int kChunks = kRowBytes / 16;
    static constexpr int kTileBytes = kTileRows * kRowBytes;
    // physical 16-byte chunk of logical chunk j in row r under the TMA swizzle
    __device__ static __forceinline__ int swz(int r, int j) {
        return sizeof(T) == 4 ? (j ^ (r & 7)) : (j ^ ((r >> 1) & 3));
    }
};

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void tma_load_2d_addr(uint32_t dst, const CUtensorMap* map, uint32_t bar, int32_t c0,
                                                 int32_t c1, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}

// Cluster launch control (Blackwell work stealing): ask the hardware to cancel a
// not-yet-launched CTA of this grid; the 16-byte response lands in shared memory
// and completes `bar`.  Returns the cancelled CTA's blockIdx.x or -1.
__device__ __forceinline__ void clc_try_cancel(uint32_t resp_addr, uint32_t bar_addr) {
    asm volatile("clusterlaunchcontrol.try_cancel.async.shared::cta.mbarrier::complete_tx::bytes.b128 [%0], [%1];"
                 ::"r"(resp_addr), "r"(bar_addr) : "memory");
}
__device__ __forceinline__ int clc_read(uint32_t resp_addr) {
    uint32_t valid, x;
    asm volatile(
        "{\n\t"
        ".reg .pred p1;\n\t"
        ".reg .b128 r;\n\t"
        ".reg .b32 y, z;\n\t"
        "ld.shared.b128 r, [%2];\n\t"
        "clusterlaunchcontrol.query_cancel.is_canceled.pred.b128 p1, r;\n\t"
        "selp.u32 %1, 1, 0, p1;\n\t"
        "mov.u32 %0, 0;\n\t"
        "@p1 clusterlaunchcontrol.query_cancel.get_first_ctaid.v4.b32.b128 {%0, y, z, _}, r;\n\t"
        "}\n"
        : "=r"(x), "=r"(valid) : "r"(resp_addr) : "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    return valid ? (int)x : -1;
}

// a / L for L in {15, 255} with the reciprocal hoisted to a constant: exact for
// every float in [2^-100, 2^100] (checked exhaustively on CPU, all 1.68e9 values).
template <int BITS>
__device__ __forceinline__ float div_by_levels(float a) {
    constexpr float L = BITS == 8 ? 255.0f : 15.0f;
    constexpr float y = BITS == 8 ? 0.00392156862745098f : 0.06666666666666667f;   // RN(1/L)
    float q0 = __fmul_rn(a, y);
    float r = __fmaf_rn(-L, q0, a);
    return __fmaf_rn(y, r, q0);
}

// Rare path (non-finite data, ranges outside [2^-50, 2^50]): generic IEEE
// arithmetic, kept out of line so the hot loop stays small in the I-cache.
template <int BITS>
__device__ __noinline__ float slow_row_codes(const float* v, float mn, float mx, uint32_t* u) {
    constexpr float L = BITS == 8 ? 255.0f : 15.0f;
    AffineParams p = affine_params(mn, mx, L);
#pragma unroll 1
    for (int k = 0; k < kRowElems; ++k) u[k] = code_bits(affine_quotient(v[k], p), L);
    return p.scale;
}

// The tensors of one launch: a single tensor (quantize_rows_tma_kernel) or up to kMultiMax of them
// (quantize_rows_tma_multi_kernel).  Quantizing a model is hundreds of independent matrices; one launch
// per matrix pays a prologue (barrier setup, tensor-map fetch, first-tile latency) and a tail each
// time.  The multi-tensor launch lets them share one grid: the tile index space is the concatenation
// of the tensors' tiles, the descriptors ride in the kernel parameters (tensor maps included), and
// cluster launch control balances the lot.
constexpr int kMultiMax = 16;
struct MultiArgs {
    CUtensorMap maps[kMultiMax];
    int64_t n_rows[kMultiMax];
    uint8_t* q[kMultiMax];
    float* scale[kMultiMax];
    float* zp[kMultiMax];
    int tile_base[kMultiMax + 1];     // first global tile of tensor i; [count] = total
    int count;
};

// Both describe their tensors to quantize_rows_stream the same way: locate() maps a tile of the
// launch to (tensor ti, tile within it).
struct RowsOne {
    static constexpr bool kMulti = false;
    const CUtensorMap* tmap;
    int64_t n_rows;
    uint8_t* q_out;
    float* scale_out;
    float* zp_out;
    __device__ __forceinline__ int n_tiles() const { return (int)((n_rows + kTileRows - 1) / kTileRows); }
    __device__ __forceinline__ int locate(int g, int& ti) const { ti = 0; return g; }
    __device__ __forceinline__ const CUtensorMap* map(int) const { return tmap; }
    __device__ __forceinline__ int64_t rows(int) const { return n_rows; }
    __device__ __forceinline__ uint8_t* q(int) const { return q_out; }
    __device__ __forceinline__ float* scale(int) const { return scale_out; }
    __device__ __forceinline__ float* zp(int) const { return zp_out; }
};
struct RowsMulti {
    static constexpr bool kMulti = true;
    const MultiArgs& a;
    __device__ __forceinline__ int n_tiles() const { return a.tile_base[a.count]; }
    __device__ __forceinline__ int locate(int g, int& ti) const {
        ti = 0;
        while (ti + 1 < a.count && g >= a.tile_base[ti + 1]) ++ti;
        return g - a.tile_base[ti];
    }
    __device__ __forceinline__ const CUtensorMap* map(int ti) const { return &a.maps[ti]; }
    __device__ __forceinline__ int64_t rows(int ti) const { return a.n_rows[ti]; }
    __device__ __forceinline__ uint8_t* q(int ti) const { return a.q[ti]; }
    __device__ __forceinline__ float* scale(int ti) const { return a.scale[ti]; }
    __device__ __forceinline__ float* zp(int ti) const { return a.zp[ti]; }
};

// How a stream launch orders itself against its neighbours on the stream (programmatic dependent launch; the
// argument is in common.cuh, next to pdl_wait).  kWaitFirst: wait for the previous kernel before the first global
// access.  Without it the launch was released early by the previous multi-tensor launch of the same call, loads at
// once and waits for that launch before it exits.  kReleaseNext: the next launch is the next multi-tensor launch of
// the same call; let it start as soon as every CTA of this one has started (or been taken over) and is past its wait.
constexpr int kWaitFirst = 1, kReleaseNext = 2;

// Blockwise (convention A) row stream, one CTA per tile of the launch: resident CTAs steal the
// not-yet-launched ones (cluster launch control).
template <typename T, int BITS, bool PACK, typename Src>
__device__ __forceinline__ void quantize_rows_stream(const Src& src, int log2_lanes_per_block, int pdl) {
    using RL = RowLayout<T>;
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t full_bar[kStages], empty_bar[kStages], clc_bar;
    __shared__ uint32_t dep_scratch[kTmaThreads / 32];           // see mbar_arrive_after_loads
    __shared__ __align__(16) uint4 clc_resp;
    __shared__ int tile_of_stage[kStages], tens_of_stage[kStages];

    const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;       // SWIZZLE_128B atoms are 1 KB
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_tiles = src.n_tiles();

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], kConsumerWarps); }
        mbar_init(&clc_bar, 1);
        fence_barrier_init();
    }
    __syncthreads();
    if (pdl & kWaitFirst) pdl_wait();                      // the set-up above may overlap the previous kernel's tail
    if (pdl & kReleaseNext) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp == kConsumerWarps) {
        // ===== producer warp: one lane streams tiles into the ring =====
        if (lane == 0) {
            if (!Src::kMulti) prefetch_tensormap(src.map(0));
            // evict-normal, not evict-first, although every tile is read once: measured 8 % faster on the
            // bench step (profiles/INDEX.md, r03)
            const uint64_t policy = policy_evict_normal();
            int cta = blockIdx.x;          // this CTA's own tile first, then stolen ones
            uint32_t clc_phase = 0;
            for (int i = 0;; ++i) {
                const int s = i % kStages;
                const uint32_t ph = (i / kStages) & 1;
                mbar_wait(&empty_bar[s], ph ^ 1);
                const bool live = cta >= 0 && cta < n_tiles;
                if (!live) { tile_of_stage[s] = -1; mbar_arrive(&full_bar[s]); break; }
                int ti;
                const int t = src.locate(cta, ti);
                tile_of_stage[s] = t;
                if (Src::kMulti) tens_of_stage[s] = ti;
                mbar_arrive_expect_tx(&full_bar[s], RL::kTileBytes);
                tma_load_2d_addr(smem + s * RL::kTileBytes, src.map(ti), smem_u32(&full_bar[s]), 0, t * kTileRows, policy);
                mbar_arrive_expect_tx(&clc_bar, 16);
                clc_try_cancel(smem_u32(&clc_resp), smem_u32(&clc_bar));
                mbar_wait(&clc_bar, clc_phase);
                clc_phase ^= 1;
                cta = clc_read(smem_u32(&clc_resp));
            }
        }
        if (!(pdl & kWaitFirst)) pdl_wait();               // our completion implies the previous launch's
        return;
    }

    // ===== consumers: thread `tid` owns row `tid` of every tile =====
    const int lpb_mask = (1 << log2_lanes_per_block) - 1;
    const uint32_t row_off = tid * RL::kRowBytes;
    for (int i = 0;; ++i) {
        const int s = i % kStages;
        const uint32_t ph = (i / kStages) & 1;
        mbar_wait(&full_bar[s], ph);
        const int t = *reinterpret_cast<volatile int*>(&tile_of_stage[s]);
        if (t < 0) break;
        const int ti = Src::kMulti ? *reinterpret_cast<volatile int*>(&tens_of_stage[s]) : 0;

        float v[kRowElems];
        const uint32_t row = smem + s * RL::kTileBytes + row_off;
#pragma unroll
        for (int j = 0; j < RL::kChunks; ++j) {
            uint4 c = lds128(row + (RL::swz(tid, j) << 4));
            if (sizeof(T) == 4) {
                v[4 * j + 0] = __uint_as_float(c.x); v[4 * j + 1] = __uint_as_float(c.y);
                v[4 * j + 2] = __uint_as_float(c.z); v[4 * j + 3] = __uint_as_float(c.w);
            } else {
                const T* e = reinterpret_cast<const T*>(&c);
#pragma unroll
                for (int k = 0; k < 8; ++k) v[8 * j + k] = to_f32(e[k]);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive_after_loads(&empty_bar[s], row_dep<T>(v), &dep_scratch[warp]);     // stage can be refilled while we compute

        const int64_t grow = (int64_t)t * kTileRows + tid;      // row within the tensor
        const bool row_ok = grow < src.rows(ti);
        uint32_t u[kRowElems];
        float m0[4], m1[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { m0[k] = v[k]; m1[k] = v[k]; }
#pragma unroll
        for (int k = 4; k < kRowElems; ++k) { m0[k & 3] = min_nan(m0[k & 3], v[k]); m1[k & 3] = max_nan(m1[k & 3], v[k]); }
        float mn = min_nan(min_nan(m0[0], m0[1]), min_nan(m0[2], m0[3]));
        float mx = max_nan(max_nan(m1[0], m1[1]), max_nan(m1[2], m1[3]));
        for (int o = 1; o <= lpb_mask; o <<= 1) {
            mn = min_nan(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        // quantization.py:195-196 / :205: degenerate range rule, scale = range / L
        const float mx2 = (mx == mn) ? __fadd_rn(mn, 1e-6f) : mx;
        const float range = __fsub_rn(mx2, mn);
        // range in [2^-50, 2^50] (false for NaN/inf): constant-reciprocal divide and
        // hoisted-reciprocal quotients are exact, and x in [mn, mx] makes the clamp a no-op
        const bool fast = range >= 8.881784197001252e-16f && range <= 1125899906842624.0f;
        float scale;
        if (__all_sync(0xffffffffu, fast)) {
            scale = div_by_levels<BITS>(range);
            const float rcp = __frcp_rn(scale);
            const float nscale = -scale;
#pragma unroll
            for (int k = 0; k < kRowElems; ++k) {
                const float d = __fsub_rn(v[k], mn);
                const float q0 = __fmul_rn(d, rcp);
                const float r = __fmaf_rn(nscale, q0, d);
                u[k] = __float_as_uint(__fadd_rn(__fmaf_rn(rcp, r, q0), kMagic));
            }
        } else {
            // copies keep v[] / u[] in registers on the hot path (only these temporaries live on the stack)
            float vs[kRowElems];
            uint32_t us[kRowElems];
#pragma unroll
            for (int k = 0; k < kRowElems; ++k) vs[k] = v[k];
            scale = slow_row_codes<BITS>(vs, mn, mx, us);
#pragma unroll
            for (int k = 0; k < kRowElems; ++k) u[k] = us[k];
        }
        if (row_ok && (lane & lpb_mask) == 0) {
            const int64_t b = grow >> log2_lanes_per_block;
            src.scale(ti)[b] = scale;
            src.zp(ti)[b] = mn;
        }
        if (row_ok) {
            if (BITS == 4 && PACK) {
                uint4 o;
                o.x = pack_nibbles8<kConvA>(u + 0);  o.y = pack_nibbles8<kConvA>(u + 8);
                o.z = pack_nibbles8<kConvA>(u + 16); o.w = pack_nibbles8<kConvA>(u + 24);
                __stcs(reinterpret_cast<uint4*>(src.q(ti) + grow * 16), o);
            } else {
                uint32_t w[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) w[k] = pack_bytes4<kConvA, BITS>(u[4 * k], u[4 * k + 1], u[4 * k + 2], u[4 * k + 3]);
                uint4* dst = reinterpret_cast<uint4*>(src.q(ti) + grow * 32);
                __stcs(dst, make_uint4(w[0], w[1], w[2], w[3]));
                __stcs(dst + 1, make_uint4(w[4], w[5], w[6], w[7]));
            }
        }
    }
    if (!(pdl & kWaitFirst)) pdl_wait();
}

template <typename T, int BITS, bool PACK>
__global__ void __launch_bounds__(kTmaThreads, 2)
quantize_rows_tma_kernel(const __grid_constant__ CUtensorMap tmap, int64_t n_rows, int log2_lanes_per_block,
                         uint8_t* __restrict__ q_out, float* __restrict__ scale_out, float* __restrict__ zp_out) {
    quantize_rows_stream<T, BITS, PACK>(RowsOne{&tmap, n_rows, q_out, scale_out, zp_out}, log2_lanes_per_block, kWaitFirst);
}

template <typename T, int BITS, bool PACK>
__global__ void __launch_bounds__(kTmaThreads, 2)
quantize_rows_tma_multi_kernel(const __grid_constant__ MultiArgs a, int log2_lanes_per_block, int pdl) {
    quantize_rows_stream<T, BITS, PACK>(RowsMulti{a}, log2_lanes_per_block, pdl);
}

// --------------------------------------------------------------------------
// 2a. TENSOR mode in ONE launch: reduce, grid barrier, quantize from shared memory / L2
// --------------------------------------------------------------------------
// Per-tensor parameters need the global min/max before the first code can be written, so the
// tensor is needed twice.  Two launches re-read all of it; here one persistent CTA per SM
//   phase 1  streams its contiguous share of 16 KB tiles through shared memory for min/max and
//            KEEPS the first R tiles there (R = all of them when the share fits: one HBM read),
//   barrier  publishes its partial min/max, arrives at a grid-wide counter, waits for the others
//            (all CTAs are resident: one per SM, grid <= #SMs, cooperative launch),
//   phase 2  quantizes the resident tiles straight from shared memory while the producer warp
//            re-streams the other tiles newest-first (they were loaded with L2 evict_last, so
//            most of them are still in the 126 MB L2).
// The counters live in the workspace header, which must be zero before the first call and is
// left zero by every call (include/quanta_b200.h).
constexpr int kFRows = 128;                       // rows per tile = threads per consumer group
constexpr int kFGroups = 4;                       // consumer groups; a ring slot always belongs to one group
constexpr int kFConsumers = kFRows * kFGroups;
constexpr int kFThreads = kFConsumers + 32;
constexpr int kFMaxSlots = 32;
constexpr int kWsArriveIdx = 8, kWsDoneIdx = 9;   // grid-barrier counters (ints) in the workspace header
constexpr int kWsErrPtrIdx = 12;                  // ints 12-13: address of a host-mapped int32 error flag (0 = none)
constexpr unsigned int kBarrierSpinLimit = 1u << 22;      // ~1 s of polling; a healthy barrier takes microseconds

// The grid barrier did not complete (the header was not zero before the call, or the grid is not co-resident).
// Instead of killing the context, report through the caller's host-mapped flag (include/quanta_b200.h), leave
// the counters zero for the next call and carry on: the results of THIS call are garbage, the host wrapper
// raises on its next entry.
__device__ __noinline__ void barrier_timeout(float* ws) {
    unsigned int* h = reinterpret_cast<unsigned int*>(ws);
    const unsigned long long flag = *reinterpret_cast<volatile unsigned long long*>(h + kWsErrPtrIdx);
    if (flag != 0ull) {
        *reinterpret_cast<volatile int*>(flag) = 1;
        __threadfence_system();
    }
    *reinterpret_cast<volatile unsigned int*>(h + kWsArriveIdx) = 0u;
    *reinterpret_cast<volatile unsigned int*>(h + kWsDoneIdx) = 0u;
    __threadfence();
}

template <typename T>
__device__ __forceinline__ void load_row32(uint32_t row_addr, int r, float* v) {
    using RL = RowLayout<T>;
#pragma unroll
    for (int j = 0; j < RL::kChunks; ++j) {
        uint4 c = lds128(row_addr + (RL::swz(r, j) << 4));
        if (sizeof(T) == 4) {
            v[4 * j + 0] = __uint_as_float(c.x); v[4 * j + 1] = __uint_as_float(c.y);
            v[4 * j + 2] = __uint_as_float(c.z); v[4 * j + 3] = __uint_as_float(c.w);
        } else {
            const T* e = reinterpret_cast<const T*>(&c);
#pragma unroll
            for (int k = 0; k < 8; ++k) v[8 * j + k] = to_f32(e[k]);
        }
    }
}

template <typename T, int BITS, bool PACK, int CONV>
__global__ void __launch_bounds__(kFThreads, 1)
quantize_tensor_fused_kernel(const __grid_constant__ CUtensorMap tmap, const T* __restrict__ x, int64_t n,
                             int64_t n_rows, int nslots, int ring_min, uint8_t* __restrict__ q_out,
                             float* __restrict__ scale_out, float* __restrict__ zp_out, float* ws) {
    using RL = RowLayout<T>;
    constexpr int kTileBytes = kFRows * RL::kRowBytes;
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t full_bar[kFMaxSlots], empty_bar[kFMaxSlots];
    __shared__ uint32_t dep_scratch[kFThreads / 32];             // see mbar_arrive_after_loads
    __shared__ float red_mn[kFConsumers / 32], red_mx[kFConsumers / 32];

    const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_tiles = (int)((n_rows + kFRows - 1) / kFRows);
    const int G = (int)gridDim.x, c = (int)blockIdx.x;
#ifdef QUANTA_FUSED_TRACE
    long long tr[8]; unsigned long long g0, g1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g0));
    tr[0] = clock64();
#define FTRACE(i) tr[i] = clock64()
#else
#define FTRACE(i) do { } while (0)
#endif
    const int t0 = (int)((int64_t)n_tiles * c / G), t1 = (int)((int64_t)n_tiles * (c + 1) / G);
    const int cnt = t1 - t0;
    const int R = cnt <= nslots ? cnt : nslots - ring_min;      // resident tiles
    const int ns = cnt - R;                                     // streamed twice
    const int ring = ns > 0 ? ring_min : kFGroups;              // multiple of kFGroups: slot -> group is fixed
    const int K = ns < kFGroups ? ns : kFGroups;                // newest streamed tiles, kept in registers over the barrier

    if (tid == 0) {
        for (int s2 = 0; s2 < nslots; ++s2) { mbar_init(&full_bar[s2], 1); mbar_init(&empty_bar[s2], kFRows / 32); }
        fence_barrier_init();
    }
    __syncthreads();

    if (warp == kFConsumers / 32) {
        // ===== producer: residents first, then the ring (phase 1 in order, phase 2 newest first) =====
        if (lane == 0) {
            prefetch_tensormap(&tmap);
            const uint64_t pol_once = policy_evict_first(), pol_again = policy_evict_last();
            for (int j = 0; j < R; ++j) {
                mbar_arrive_expect_tx(&full_bar[j], kTileBytes);
                tma_load_2d_addr(smem + j * kTileBytes, &tmap, smem_u32(&full_bar[j]), 0, (t0 + j) * kFRows, pol_once);
            }
            for (int m = 0; m < 2 * ns - K; ++m) {
                const int u = m / ring, slot = R + (m - u * ring);
                if (u > 0) mbar_wait(&empty_bar[slot], (uint32_t)((u & 1) ^ 1));
                const int t = m < ns ? t0 + R + m : t1 - 1 - K - (m - ns);
                mbar_arrive_expect_tx(&full_bar[slot], kTileBytes);
                tma_load_2d_addr(smem + slot * kTileBytes, &tmap, smem_u32(&full_bar[slot]), 0, t * kFRows,
                                 m < ns ? pol_again : pol_once);
            }
        }
        return;
    }

    // ===== consumers: group g owns the items it can reach with a fixed slot -> group map =====
    const int group = tid >> 7, r = tid & (kFRows - 1);
    const uint32_t row_off = (uint32_t)r * RL::kRowBytes;
    constexpr float L = BITS == 8 ? 255.0f : 15.0f;
    constexpr float Q = BITS == 8 ? 127.0f : 7.0f;

    FTRACE(1);
    // ---- phase 1: min / max ----
    float m0[4], m1[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { m0[k] = __int_as_float(0x7f800000); m1[k] = __int_as_float(0xff800000); }
    for (int i = group; i < R; i += kFGroups) {
        mbar_wait(&full_bar[i], 0);
        if ((int64_t)(t0 + i) * kFRows + r < n_rows) {
            float v[kRowElems];
            load_row32<T>(smem + i * kTileBytes + row_off, r, v);
#pragma unroll
            for (int k = 0; k < kRowElems; ++k) { m0[k & 3] = min_nan(m0[k & 3], v[k]); m1[k & 3] = max_nan(m1[k & 3], v[k]); }
        }
    }
    // ring use m is consumed by group (R + m) % kFGroups
    const int mfirst = (group - R % kFGroups + kFGroups) % kFGroups;
    // The row of the group's LAST streamed tile stays in `vk` across the grid barrier: the K newest
    // tiles (one per group) are quantized from registers and never fetched again.
    float vk[kRowElems];
#pragma unroll
    for (int k = 0; k < kRowElems; ++k) vk[k] = 0.0f;
    int keep_m = -1;
    for (int m = mfirst; m < ns; m += kFGroups) {
        const int u = m / ring, slot = R + (m - u * ring);
        mbar_wait(&full_bar[slot], (uint32_t)(u & 1));
        load_row32<T>(smem + slot * kTileBytes + row_off, r, vk);
        __syncwarp();
        if (lane == 0) mbar_arrive_after_loads(&empty_bar[slot], row_dep<T>(vk), &dep_scratch[warp]);
        if ((int64_t)(t0 + R + m) * kFRows + r < n_rows) {
#pragma unroll
            for (int k = 0; k < kRowElems; ++k) { m0[k & 3] = min_nan(m0[k & 3], vk[k]); m1[k & 3] = max_nan(m1[k & 3], vk[k]); }
        }
        keep_m = m;
    }
    float mn = min_nan(min_nan(m0[0], m0[1]), min_nan(m0[2], m0[3]));
    float mx = max_nan(max_nan(m1[0], m1[1]), max_nan(m1[2], m1[3]));
    // elements past the last full 32-element row (the tail kernel quantizes them)
    if (c == 0) {
        const int64_t j = n_rows * kRowElems + tid;
        if (j < n) { const float f = to_f32(x[j]); mn = min_nan(mn, f); mx = max_nan(mx, f); }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = min_nan(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0) { red_mn[warp] = mn; red_mx[warp] = mx; }
    asm volatile("bar.sync 1, %0;" ::"n"(kFConsumers) : "memory");

    FTRACE(2);
    // ---- grid barrier: warp 0 publishes the CTA's partial, waits for all CTAs, reduces their partials ----
    float* pmin = ws + kWsHeaderFloats + 64;
    float* pmax = pmin + kMaxPartialCtas;
    unsigned int* arrive = reinterpret_cast<unsigned int*>(ws) + kWsArriveIdx;
    unsigned int* done = reinterpret_cast<unsigned int*>(ws) + kWsDoneIdx;
    if (warp == 0) {
        mn = red_mn[lane & (kFConsumers / 32 - 1)]; mx = red_mx[lane & (kFConsumers / 32 - 1)];
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {
            mn = min_nan(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        if (lane == 0) {
            pmin[c] = mn; pmax[c] = mx;
            // release: the partial above is visible to whoever observes the incremented counter
            asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(arrive) : "memory");
            unsigned int seen = 0, spins = 0;
            for (;;) {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(arrive) : "memory");
                if (seen >= (unsigned int)G) break;
                if (++spins > kBarrierSpinLimit) { barrier_timeout(ws); break; }
            }
        }
        __syncwarp();
        asm volatile("fence.acq_rel.gpu;" ::: "memory");
        float v0[5], v1[5];                            // G <= 148 partials: 5 per lane, all loads in flight at once
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const int idx = lane + 32 * k;
            v0[k] = __ldcg(pmin + (idx < G ? idx : 0));
            v1[k] = __ldcg(pmax + (idx < G ? idx : 0));
        }
        mn = v0[0]; mx = v1[0];
#pragma unroll
        for (int k = 1; k < 5; ++k) { mn = min_nan(mn, v0[k]); mx = max_nan(mx, v1[k]); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mn = min_nan(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        if (lane == 0) {
            red_mn[0] = mn; red_mx[0] = mx;
            // every partial has been read by this CTA; the last CTA through leaves the counters zero
            const unsigned int old = atomicAdd(done, 1u);
            if (old == (unsigned int)(G - 1)) { *arrive = 0u; *done = 0u; }
        }
    }
    FTRACE(3);
    asm volatile("bar.sync 1, %0;" ::"n"(kFConsumers) : "memory");
    mn = red_mn[0]; mx = red_mx[0];

    ElemParams gp{0.f, 1.f, 0.f};
    float sc, z, rr; bool close;
    group_params<CONV>(mn, mx, BITS, &sc, &z, &rr, &close);
    const bool early = (CONV != kConvA) && close;
    if (early) { sc = 1.0f; z = mn; }                     // cpu/quantization.py:38-39
    gp.s = sc; gp.a = z; gp.r = rr;
    if (c == 0 && tid == 0) {                             // publish for the caller and the tail kernel
        scale_out[0] = sc; zp_out[0] = z;
        ws[kWsHeaderFloats] = rr;
        reinterpret_cast<int*>(ws)[0] = early ? 1 : 0;
    }

    // ---- phase 2: codes ----
    auto quantize_row = [&](const float* v, int t) {
        const int64_t grow = (int64_t)t * kFRows + r;
        if (grow >= n_rows) return;
        uint32_t u[kRowElems];
        if (CONV == kConvA && gp.r != 0.0f) {
            const float nscale = -gp.s;
#pragma unroll
            for (int k = 0; k < kRowElems; ++k) {
                const float a = __fsub_rn(v[k], gp.a);
                const float q0 = __fmul_rn(a, gp.r);
                const float rem = __fmaf_rn(nscale, q0, a);
                // rcp != 0: the range is finite, every x lies in [min, max] and the quotient in
                // [0, L + eps] — the clamp of code_bits is a no-op
                u[k] = __float_as_uint(__fadd_rn(__fmaf_rn(gp.r, rem, q0), kMagic));
            }
        } else {
#pragma unroll
            for (int k = 0; k < kRowElems; ++k) u[k] = elem_code_bits<CONV, false>(v[k], gp, L, Q);
        }
        if (BITS == 4 && PACK) {
            uint4 o;
            o.x = pack_nibbles8<CONV>(u + 0);  o.y = pack_nibbles8<CONV>(u + 8);
            o.z = pack_nibbles8<CONV>(u + 16); o.w = pack_nibbles8<CONV>(u + 24);
            if (early) o = make_uint4(0, 0, 0, 0);
            __stcs(reinterpret_cast<uint4*>(q_out + grow * 16), o);
        } else {
            uint32_t w[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) w[k] = early ? 0u : pack_bytes4<CONV, BITS>(u[4 * k], u[4 * k + 1], u[4 * k + 2], u[4 * k + 3]);
            uint4* dst = reinterpret_cast<uint4*>(q_out + grow * 32);
            __stcs(dst, make_uint4(w[0], w[1], w[2], w[3]));
            __stcs(dst + 1, make_uint4(w[4], w[5], w[6], w[7]));
        }
    };
    FTRACE(4);
    if (keep_m >= ns - K && keep_m >= 0) quantize_row(vk, t0 + R + keep_m);       // from registers
    FTRACE(5);
    // resident tiles (shared memory) and re-streamed tiles (L2, newest first) alternate, so the L2
    // latency of the ring hides behind the resident tiles' arithmetic.  Phase-2 ring uses continue the
    // numbering: use m = ns + k re-reads tile t1 - 1 - K - k.
    const int m_end = 2 * ns - K;
    int i2 = group;
    int m2 = ns + ((group - (R + ns) % kFGroups + kFGroups) % kFGroups);
    while (i2 < R || m2 < m_end) {
        if (i2 < R) {
            float v[kRowElems];
            load_row32<T>(smem + i2 * kTileBytes + row_off, r, v);
            quantize_row(v, t0 + i2);
            i2 += kFGroups;
        }
        if (m2 < m_end) {
            const int u = m2 / ring, slot = R + (m2 - u * ring);
            mbar_wait(&full_bar[slot], (uint32_t)(u & 1));
            float v[kRowElems];
            load_row32<T>(smem + slot * kTileBytes + row_off, r, v);
            __syncwarp();
            if (lane == 0) mbar_arrive_after_loads(&empty_bar[slot], row_dep<T>(v), &dep_scratch[warp]);          // refill while we compute
            quantize_row(v, t1 - 1 - K - (m2 - ns));
            m2 += kFGroups;
        }
    }
#ifdef QUANTA_FUSED_TRACE
    FTRACE(6);
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
    if (tid == 0 && (c == 0 || c == G - 1))
        printf("cta %d cnt %d R %d ns %d: init %lld ph1 %lld arrive+spin %lld reduce %lld resident %lld streamed %lld | total %lld cyc, %llu ns (start %llu)\n",
               c, cnt, R, ns, tr[1] - tr[0], tr[2] - tr[1], tr[3] - tr[2], tr[4] - tr[3], tr[5] - tr[4], tr[6] - tr[5], tr[6] - tr[0], g1 - g0, g0);
#endif
}

// --------------------------------------------------------------------------
// 2a'. DIM0 mode (per_channel=True, convention A) in ONE launch
// --------------------------------------------------------------------------
// Same skeleton as the per-tensor kernel, over 2-D tiles of the matrix: a tile is [128 rows x 32
// columns], tiles are numbered down the rows of a 32-column strip first, and a CTA's contiguous
// tile range touches a few strips.  Phase 1 reduces columns (lane = column, a warp walks 32 rows:
// conflict-free under the TMA swizzle) into per-strip tables in shared memory and publishes them;
// after the grid barrier every CTA combines, for each of ITS strips, the partials of the CTAs that
// share the strip, derives the 32 columns' parameters once into shared memory, and phase 2
// quantizes row-per-thread with broadcast parameter reads.
constexpr int kD0MaxStrips = 16;                 // strips per CTA the shared parameter table can hold
constexpr int kD0SlotFloats = 64;                // one partial: 32 column minima + 32 maxima (as ordered keys)

// float <-> unsigned key whose integer order is the float order (-0.0 < +0.0); NaN maps to the
// extreme that wins the reduction, so min/max propagate NaN like torch.min / torch.max
__device__ __forceinline__ uint32_t key_of(float f, bool for_min) {
    const uint32_t b = __float_as_uint(f);
    if (f != f) return for_min ? 0u : 0xFFFFFFFFu;
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float float_of_key(uint32_t k) {
    if (k == 0u || k == 0xFFFFFFFFu) return __int_as_float(0x7fc00000);        // only NaN maps there
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

struct Dim0Geom {
    int tps;            // tiles per strip = ceil(rows / 128)
    int n_tiles;
    int max_strips;     // partial slots per CTA
};
// first tile of CTA c: floor(n_tiles * c / G) in 32-bit arithmetic (tq = n_tiles / G, trem = n_tiles % G)
struct Dim0Split { int G, tq, trem; };
__device__ __forceinline__ int d0_first_tile(int c, const Dim0Split& sp) { return sp.tq * c + (sp.trem * c) / sp.G; }
__device__ __forceinline__ int d0_cta_of_tile(int t, const Dim0Split& sp) {
    int c = sp.tq > 0 ? t / (sp.tq + 1) : 0;             // never above the answer: first_tile(c) <= (tq + 1) * c
    if (c > sp.G - 1) c = sp.G - 1;
    while (c + 1 < sp.G && d0_first_tile(c + 1, sp) <= t) ++c;
    return c;
}

// 4 consecutive columns (quad cq) of tile row `row`
template <typename T>
__device__ __forceinline__ void d0_load4(uint32_t tile_addr, int row, int cq, float* f) {
    using RL = RowLayout<T>;
    if (sizeof(T) == 4) {
        const uint4 v = lds128(tile_addr + (uint32_t)row * RL::kRowBytes + ((uint32_t)RL::swz(row, cq) << 4));
        f[0] = __uint_as_float(v.x); f[1] = __uint_as_float(v.y); f[2] = __uint_as_float(v.z); f[3] = __uint_as_float(v.w);
    } else {
        uint2 v;
        const uint32_t a = tile_addr + (uint32_t)row * RL::kRowBytes + ((uint32_t)RL::swz(row, cq >> 1) << 4) + (uint32_t)(cq & 1) * 8u;
        asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
        const T* e2 = reinterpret_cast<const T*>(&v);
#pragma unroll
        for (int j = 0; j < 4; ++j) f[j] = to_f32(e2[j]);
    }
}
template <int BITS, bool PACK>
__device__ __forceinline__ void d0_stage4(uint32_t stage, int row, int cq, const uint32_t* u) {
    if (BITS == 4 && PACK) {
        const uint32_t h = (((u[3] * 16u + u[2]) * 16u + u[1]) * 16u + u[0]) - kMagicBits * 0x1111u;
        asm volatile("st.shared.b16 [%0], %1;" ::"r"(stage + (uint32_t)row * 16u + (uint32_t)cq * 2u), "h"((unsigned short)h) : "memory");
    } else {
        const uint32_t w = pack_bytes4<kConvA, BITS>(u[0], u[1], u[2], u[3]);
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(stage + (uint32_t)row * 32u + (uint32_t)cq * 4u), "r"(w) : "memory");
    }
}
// rare: a tile with a column whose scale is outside [2^-60, 2^60] (constant-zero columns, inf/NaN):
// generic arithmetic with true divides, out of line (scalar arguments only, so nothing of the hot path
// is forced into local memory)
template <typename T, int BITS, bool PACK>
__device__ __noinline__ void d0_tile_slow(uint32_t tile_addr, uint32_t stage, int row_base, int cq, float4 a4, float4 s4,
                                          float4 r4) {
    constexpr float L = BITS == 8 ? 255.0f : 15.0f;
    const ElemParams ep[4] = {{a4.x, s4.x, r4.x}, {a4.y, s4.y, r4.y}, {a4.z, s4.z, r4.z}, {a4.w, s4.w, r4.w}};
#pragma unroll 1
    for (int i = 0; i < 8; ++i) {
        const int row = row_base + 4 * i;
        float f[4];
        d0_load4<T>(tile_addr, row, cq, f);
        uint32_t u[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) u[j] = elem_code_bits<kConvA>(f[j], ep[j], L, 0.0f);
        d0_stage4<BITS, PACK>(stage, row, cq, u);
    }
}

template <typename T, int BITS, bool PACK>
__global__ void __launch_bounds__(kFThreads, 1)
quantize_dim0_fused_kernel(const __grid_constant__ CUtensorMap tmap, int64_t rows, int64_t cols, Dim0Geom geo,
                           int nslots, int ring_min, uint8_t* __restrict__ q_out, float* __restrict__ scale_out,
                           float* __restrict__ zp_out, float* ws) {
    using RL = RowLayout<T>;
    constexpr int kTileBytes = kFRows * RL::kRowBytes;
    constexpr float L = BITS == 8 ? 255.0f : 15.0f;
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t full_bar[kFMaxSlots], empty_bar[kFMaxSlots];
    __shared__ uint32_t dep_scratch[kFThreads / 32];             // see mbar_arrive_after_loads
    __shared__ uint32_t skey[kD0MaxStrips][2][32];                 // per local strip: column min / max keys
    __shared__ __align__(16) float sparam[kD0MaxStrips][3][32];    // per strip: zero point (min) | scale | rcp of 32 columns

    const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int G = (int)gridDim.x, c = (int)blockIdx.x;
    const int n_tiles = geo.n_tiles, tps = geo.tps;
#ifdef QUANTA_FUSED_TRACE
    long long tr[8];
    tr[0] = clock64();
#endif
    const Dim0Split sp{G, n_tiles / G, n_tiles % G};
    const int t0 = d0_first_tile(c, sp), t1 = d0_first_tile(c + 1, sp);
    const int cnt = t1 - t0;
    const int R = cnt <= nslots ? cnt : nslots - ring_min;
    const int ns = cnt - R;
    const int ring = ns > 0 ? ring_min : kFGroups;
    constexpr int K = 0;                        // no register-held tiles here (keeps phase 2 to ONE inlined tile body)
    const int s_first = t0 / tps;
    const int nls = (t1 - 1) / tps - s_first + 1;                  // local strips of this CTA (<= geo.max_strips)

    if (tid == 0) {
        for (int s2 = 0; s2 < nslots; ++s2) { mbar_init(&full_bar[s2], 1); mbar_init(&empty_bar[s2], kFRows / 32); }
        fence_barrier_init();
    }
    for (int i = tid; i < nls * 32; i += kFThreads) { skey[i >> 5][0][i & 31] = 0xFFFFFFFFu; skey[i >> 5][1][i & 31] = 0u; }
    __syncthreads();

    if (warp == kFConsumers / 32) {
        if (lane == 0) {
            prefetch_tensormap(&tmap);
            const uint64_t pol_once = policy_evict_first(), pol_again = policy_evict_last();
            auto load = [&](int slot, int t, uint64_t pol) {
                const int strip = t / tps, rb = t - strip * tps;
                mbar_arrive_expect_tx(&full_bar[slot], kTileBytes);
                tma_load_2d_addr(smem + slot * kTileBytes, &tmap, smem_u32(&full_bar[slot]), strip * kRowElems, rb * kFRows, pol);
            };
            for (int j = 0; j < R; ++j) load(j, t0 + j, pol_once);
            for (int m = 0; m < 2 * ns - K; ++m) {
                const int u = m / ring, slot = R + (m - u * ring);
                if (u > 0) mbar_wait(&empty_bar[slot], (uint32_t)((u & 1) ^ 1));
                load(slot, m < ns ? t0 + R + m : t1 - 1 - K - (m - ns), m < ns ? pol_again : pol_once);
            }
        }
        return;
    }

    const int group = tid >> 7, r = tid & (kFRows - 1), gw = (tid >> 5) & 3;       // gw: warp within the group
    // Thread mapping of both phases: lane = (column quad cq, row phase rp); in step i the warp covers rows
    // 32*gw + 4*i + rp, i = 0..7 — one 16-byte chunk per lane, 8 lanes per 128-byte tile row: conflict-free
    // under the TMA swizzle, and a thread only ever needs the parameters of ITS 4 columns.
    const int cq = lane & 7, rp = lane >> 3;
    auto load4 = [&](uint32_t tile_addr, int row, float* f) { d0_load4<T>(tile_addr, row, cq, f); };

    // ---- phase 1: column min / max ----
    float cmn[4], cmx[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { cmn[j] = __int_as_float(0x7f800000); cmx[j] = __int_as_float(0xff800000); }
    int cur_ls = -1;
    auto flush = [&]() {
        if (cur_ls >= 0) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                atomicMin(&skey[cur_ls][0][4 * cq + j], key_of(cmn[j], true));
                atomicMax(&skey[cur_ls][1][4 * cq + j], key_of(cmx[j], false));
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) { cmn[j] = __int_as_float(0x7f800000); cmx[j] = __int_as_float(0xff800000); }
    };
    auto reduce_tile = [&](uint32_t tile_addr, int t) -> uint32_t {
        const int strip = t / tps, rb = t - strip * tps;
        if (strip - s_first != cur_ls) { flush(); cur_ls = strip - s_first; }
        const int64_t row0 = (int64_t)rb * kFRows;
        uint32_t dep = 0;                                      // one word of every load (mbar_arrive_after_loads)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int row = 32 * gw + 4 * i + rp;
            float f[4];
            load4(tile_addr, row, f);
            dep ^= __float_as_uint(f[0]);
            if (row0 + row < rows) {                               // rows past the end are TMA zero fill
#pragma unroll
                for (int j = 0; j < 4; ++j) { cmn[j] = min_nan(cmn[j], f[j]); cmx[j] = max_nan(cmx[j], f[j]); }
            }
        }
        return dep;
    };
    for (int i = group; i < R; i += kFGroups) {
        mbar_wait(&full_bar[i], 0);
        reduce_tile(smem + i * kTileBytes, t0 + i);
    }
    const int mfirst = (group - R % kFGroups + kFGroups) % kFGroups;
    for (int m = mfirst; m < ns; m += kFGroups) {
        const int u = m / ring, slot = R + (m - u * ring);
        mbar_wait(&full_bar[slot], (uint32_t)(u & 1));
        const uint32_t dep = reduce_tile(smem + slot * kTileBytes, t0 + R + m);
        __syncwarp();
        if (lane == 0) mbar_arrive_after_loads(&empty_bar[slot], dep, &dep_scratch[warp]);
    }
    flush();
    asm volatile("bar.sync 1, %0;" ::"n"(kFConsumers) : "memory");

    FTRACE(2);
    // ---- publish this CTA's strip tables, grid barrier ----
    uint32_t* part = reinterpret_cast<uint32_t*>(ws + kWsHeaderFloats) + cols +
                     (size_t)c * geo.max_strips * kD0SlotFloats;
    for (int i = tid; i < nls * kD0SlotFloats; i += kFConsumers)
        part[i] = skey[i >> 6][(i >> 5) & 1][i & 31];
    __threadfence();
    asm volatile("bar.sync 1, %0;" ::"n"(kFConsumers) : "memory");
    unsigned int* arrive = reinterpret_cast<unsigned int*>(ws) + kWsArriveIdx;
    unsigned int* done = reinterpret_cast<unsigned int*>(ws) + kWsDoneIdx;
    if (tid == 0) {
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(arrive) : "memory");
        unsigned int seen = 0, spins = 0;
        for (;;) {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(arrive) : "memory");
            if (seen >= (unsigned int)G) break;
            if (++spins > kBarrierSpinLimit) { barrier_timeout(ws); break; }
        }
        __threadfence();
    }
    asm volatile("bar.sync 1, %0;" ::"n"(kFConsumers) : "memory");

    FTRACE(3);
    // ---- parameters of every column of every strip this CTA touches ----
    for (int i = tid; i < nls * 32; i += kFConsumers) {
        const int ls = i >> 5, col = i & 31;
        const int strip = s_first + ls;
        const int ta = strip * tps, tb = ta + tps - 1;
        const int c_lo = d0_cta_of_tile(ta, sp), c_hi = d0_cta_of_tile(tb, sp);
        uint32_t kmn = 0xFFFFFFFFu, kmx = 0u;
        for (int cc = c_lo; cc <= c_hi; ++cc) {
            const int ls2 = strip - d0_first_tile(cc, sp) / tps;
            const uint32_t* pp = reinterpret_cast<const uint32_t*>(ws + kWsHeaderFloats) + cols +
                                 ((size_t)cc * geo.max_strips + ls2) * kD0SlotFloats;
            kmn = min(kmn, __ldcg(pp + col));
            kmx = max(kmx, __ldcg(pp + 32 + col));
        }
        const AffineParams ap = affine_params(float_of_key(kmn), float_of_key(kmx), L);
        sparam[ls][0][col] = ap.mn; sparam[ls][1][col] = ap.scale; sparam[ls][2][col] = ap.rcp;
        if (c == c_lo) { scale_out[(int64_t)strip * 32 + col] = ap.scale; zp_out[(int64_t)strip * 32 + col] = ap.mn; }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(kFConsumers) : "memory");
    if (tid == 0) {
        const unsigned int old = atomicAdd(done, 1u);
        if (old == (unsigned int)(G - 1)) { *arrive = 0u; *done = 0u; }
    }

    // ---- phase 2: codes.  Same (column quad, row phase) mapping with the 4 columns' parameters in
    // registers; the 4 codes of a step go to a [128 rows x 32 B] staging tile of the group, which is
    // then written out row per thread: one full 32-byte sector per store. ----
    constexpr int kStageRow = (BITS == 4 && PACK) ? 16 : 32;
    const uint32_t stage = smem + (uint32_t)nslots * kTileBytes + (uint32_t)group * (kFRows * 32);
    float pa[4], ps[4], pr[4];
    int par_ls = -1;
    bool slow = false;
    float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f), s4 = a4, r4 = a4;
    auto quantize_tile = [&](uint32_t tile_addr, int t) {
        const int strip = t / tps;
        if (strip - s_first != par_ls) {
            par_ls = strip - s_first;
            a4 = *reinterpret_cast<const float4*>(&sparam[par_ls][0][4 * cq]);
            s4 = *reinterpret_cast<const float4*>(&sparam[par_ls][1][4 * cq]);
            r4 = *reinterpret_cast<const float4*>(&sparam[par_ls][2][4 * cq]);
            pa[0] = a4.x; pa[1] = a4.y; pa[2] = a4.z; pa[3] = a4.w;
            ps[0] = s4.x; ps[1] = s4.y; ps[2] = s4.z; ps[3] = s4.w;
            pr[0] = r4.x; pr[1] = r4.y; pr[2] = r4.z; pr[3] = r4.w;
            slow = __any_sync(0xffffffffu, pr[0] == 0.0f || pr[1] == 0.0f || pr[2] == 0.0f || pr[3] == 0.0f);
        }
        if (slow) { d0_tile_slow<T, BITS, PACK>(tile_addr, stage, 32 * gw + rp, cq, a4, s4, r4); return; }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int row = 32 * gw + 4 * i + rp;
            float f[4];
            load4(tile_addr, row, f);
            uint32_t u[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float a = __fsub_rn(f[j], pa[j]);
                const float q0 = __fmul_rn(a, pr[j]);
                const float rem = __fmaf_rn(-ps[j], q0, a);
                u[j] = __float_as_uint(__fadd_rn(__fmaf_rn(pr[j], rem, q0), kMagic));   // in [0, L]: no clamp needed
            }
            d0_stage4<BITS, PACK>(stage, row, cq, u);
        }
    };
    // staging -> global: thread r owns row r of the tile
    auto write_tile = [&](int t) {
        const int strip = t / tps, rb = t - strip * tps;
        asm volatile("bar.sync %0, %1;" ::"r"(2 + group), "n"(kFRows) : "memory");      // staging complete
        const int64_t grow = (int64_t)rb * kFRows + r;
#ifdef QUANTA_D0_NOSTORE
        if (grow < 0) {
#else
        if (grow < rows) {
#endif
            const int64_t e0 = grow * cols + (int64_t)strip * kRowElems;
            if (kStageRow == 16) {
                const uint4 o = lds128(stage + (uint32_t)r * 16u);
                __stcs(reinterpret_cast<uint4*>(q_out + (e0 >> 1)), o);
            } else {
                const uint4 o0 = lds128(stage + (uint32_t)r * 32u), o1 = lds128(stage + (uint32_t)r * 32u + 16u);
                asm volatile("st.global.cs.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                             ::"l"(q_out + e0), "r"(o0.x), "r"(o0.y), "r"(o0.z), "r"(o0.w), "r"(o1.x), "r"(o1.y), "r"(o1.z), "r"(o1.w)
                             : "memory");
            }
        }
        asm volatile("bar.sync %0, %1;" ::"r"(2 + group), "n"(kFRows) : "memory");      // staging may be overwritten
    };
    FTRACE(4);
    FTRACE(5);
    // resident tiles (shared memory) and re-streamed tiles (L2, newest first) alternate, so the ring's L2
    // latency hides behind the resident tiles' arithmetic
    const int m_end = 2 * ns;
    int i2 = group;
    int m2 = ns + ((group - (R + ns) % kFGroups + kFGroups) % kFGroups);
    bool turn = false;
#ifdef QUANTA_FUSED_TRACE
    long long tw = 0, tq = 0, ts = 0, tc;
#define FACC(acc) do { long long now = clock64(); acc += now - tc; tc = now; } while (0)
    tc = clock64();
#else
#define FACC(acc) do { } while (0)
#endif
    while (i2 < R || m2 < m_end) {
        const bool streamed = (m2 < m_end) && (turn || i2 >= R);
        turn = !turn;
        uint32_t ta; int t, slot = -1;
        if (!streamed) {
            ta = smem + i2 * kTileBytes; t = t0 + i2; i2 += kFGroups;
        } else {
            const int u = m2 / ring;
            slot = R + (m2 - u * ring);
            mbar_wait(&full_bar[slot], (uint32_t)(u & 1));
            ta = smem + slot * kTileBytes; t = t1 - 1 - (m2 - ns); m2 += kFGroups;
        }
        FACC(tw);
        quantize_tile(ta, t);
        if (slot >= 0) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[slot]);          // every lane has read its 8 chunks
        }
        FACC(tq);
        write_tile(t);
        FACC(ts);
    }
#ifdef QUANTA_FUSED_TRACE
    if (tid == 0 && c == 0) printf("dim0 phase2: wait %lld quantize %lld write %lld slow %d\n", tw, tq, ts, (int)slow);
#endif
#ifdef QUANTA_FUSED_TRACE
    FTRACE(6);
    if (tid == 0 && (c == 0 || c == G - 1))
        printf("dim0 cta %d cnt %d R %d ns %d nls %d: init %lld ph1 %lld barrier %lld params %lld regtile %lld rest %lld | total %lld\n",
               c, cnt, R, ns, nls, tr[1] - tr[0], tr[2] - tr[1], tr[3] - tr[2], tr[4] - tr[3], tr[5] - tr[4], tr[6] - tr[5], tr[6] - tr[0]);
#endif
}

// --------------------------------------------------------------------------
// 3. dim-0 quantize: thread owns 4 columns, walks down the rows
// --------------------------------------------------------------------------
template <typename T, int BITS, bool PACK, int CONV>
__global__ void __launch_bounds__(128) quantize_dim0_kernel(const T* __restrict__ x, int64_t rows, int64_t cols,
                                                            int rows_per_chunk, uint8_t* __restrict__ q_out,
                                                            const float* __restrict__ scale, const float* __restrict__ zp,
                                                            const float* __restrict__ ws) {
    pdl_wait();                                            // launched with programmatic stream serialization (launch_pdl)
    const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (c >= cols) return;
    constexpr float L = BITS == 8 ? 255.0f : 15.0f;
    constexpr float Q = BITS == 8 ? 127.0f : 7.0f;
    const bool early = (CONV != kConvA) && reinterpret_cast<const int*>(ws)[0] != 0;
    ElemParams p[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { p[j].s = scale[c + j]; p[j].a = zp[c + j]; p[j].r = (CONV == kConvA) ? ws[kWsHeaderFloats + c + j] : 0.f; }
    const int64_t r0 = (int64_t)(gridDim.y - 1 - blockIdx.y) * rows_per_chunk;   // newest-in-L2 first
    const int64_t r1 = min(rows, r0 + rows_per_chunk);
    auto load4 = [&](int64_t r, float* f) {
        if (sizeof(T) == 4) {
            float4 v = __ldcs(reinterpret_cast<const float4*>(x + r * cols + c));
            f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
        } else {
            uint2 v = __ldcs(reinterpret_cast<const uint2*>(x + r * cols + c));
            const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
            for (int j = 0; j < 4; ++j) f[j] = to_f32(e[j]);
        }
    };
    auto emit = [&](int64_t r, const float* f) {
        uint32_t u[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) u[j] = elem_code_bits<CONV>(f[j], p[j], L, Q);
        uint32_t w = early ? 0u : pack_bytes4<CONV, BITS>(u[0], u[1], u[2], u[3]);
        if (BITS == 4 && PACK) {
            // bytes b0..b3 (each <= 15) -> (b0 | b1<<4) | (b2 | b3<<4) << 8
            uint32_t t = w | (w >> 4);
            uint16_t h = (uint16_t)((t & 0xFFu) | ((t >> 8) & 0xFF00u));
            *reinterpret_cast<uint16_t*>(q_out + (r * cols + c) / 2) = h;
        } else {
            *reinterpret_cast<uint32_t*>(q_out + r * cols + c) = w;
        }
    };
    int64_t r = r0;
    for (; r + 3 < r1; r += 4) {
        float f[4][4];
#pragma unroll
        for (int k = 0; k < 4; ++k) load4(r + k, f[k]);
#pragma unroll
        for (int k = 0; k < 4; ++k) emit(r + k, f[k]);
    }
    for (; r < r1; ++r) { float f[4]; load4(r, f); emit(r, f); }
}

// --------------------------------------------------------------------------
// 4. generic fallbacks (tails, odd shapes, unaligned pointers)
// --------------------------------------------------------------------------
// One thread per PAIR of elements of the flat range [start, n); channel of
// element i is 0 (nchan == 1) or i % nchan.
template <typename T, int BITS, bool PACK, int CONV>
__global__ void __launch_bounds__(256) quantize_generic_kernel(const T* __restrict__ x, int64_t start, int64_t n,
                                                               int64_t nchan, uint8_t* __restrict__ q_out,
                                                               const float* __restrict__ scale,
                                                               const float* __restrict__ zp,
                                                               const float* __restrict__ ws) {
    pdl_wait();                                            // launched with programmatic stream serialization (launch_pdl)
    constexpr float L = BITS == 8 ? 255.0f : 15.0f;
    constexpr float Q = BITS == 8 ? 127.0f : 7.0f;
    constexpr uint32_t off = (CONV == kConvBSym) ? (BITS == 8 ? 128u : 8u) : 0u;
    const bool early = (CONV != kConvA) && reinterpret_cast<const int*>(ws)[0] != 0;
    const int64_t i0 = start + 2 * ((int64_t)blockIdx.x * blockDim.x + threadIdx.x);
    if (i0 >= n) return;
    uint32_t code[2] = {0, 0};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int64_t i = i0 + k;
        if (i < n) {
            const int64_t c = nchan == 1 ? 0 : i % nchan;
            ElemParams p{zp[c], scale[c], (CONV == kConvA) ? ws[kWsHeaderFloats + c] : 0.f};
            uint32_t u = elem_code_bits<CONV>(to_f32(x[i]), p, L, Q);
            code[k] = early ? 0u : ((u - kMagicBits + off) & 0xFFu);
        }
    }
    if (BITS == 4 && PACK) {
        q_out[i0 >> 1] = (uint8_t)(code[0] | (code[1] << 4));   // odd tail: pad nibble 0
    } else {
        q_out[i0] = (uint8_t)code[0];
        if (i0 + 1 < n) q_out[i0 + 1] = (uint8_t)code[1];
    }
}

// Blockwise, any block size: one warp per quantization block (two passes, the
// second one served by L1/L2).  PACK needs an even block.
template <typename T, int BITS, bool PACK>
__global__ void __launch_bounds__(256) quantize_block_generic_kernel(const T* __restrict__ x, int64_t nblocks,
                                                                     int64_t block, uint8_t* __restrict__ q_out,
                                                                     float* __restrict__ scale_out,
                                                                     float* __restrict__ zp_out) {
    pdl_wait();                                            // launched with programmatic stream serialization (launch_pdl)
    constexpr float L = BITS == 8 ? 255.0f : 15.0f;
    const int lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= nblocks) return;
    const T* xb = x + b * block;
    float mn = to_f32(xb[0]), mx = mn;
    for (int64_t i = lane; i < block; i += 32) { float f = to_f32(xb[i]); mn = min_nan(mn, f); mx = max_nan(mx, f); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = min_nan(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = max_nan(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    AffineParams p = affine_params(mn, mx, L);
    if (lane == 0) { scale_out[b] = p.scale; zp_out[b] = p.mn; }
    if (BITS == 4 && PACK) {
        uint8_t* qb = q_out + b * (block / 2);
        for (int64_t i = 2 * lane; i < block; i += 64) {
            uint32_t lo = code_bits(affine_quotient(to_f32(xb[i]), p), L) & 0xFu;
            uint32_t hi = code_bits(affine_quotient(to_f32(xb[i + 1]), p), L) & 0xFu;
            qb[i >> 1] = (uint8_t)(lo | (hi << 4));
        }
    } else {
        uint8_t* qb = q_out + b * block;
        for (int64_t i = lane; i < block; i += 32) qb[i] = (uint8_t)(code_bits(affine_quotient(to_f32(xb[i]), p), L) & 0xFFu);
    }
}

// --------------------------------------------------------------------------
// host side
// --------------------------------------------------------------------------
template <typename T> struct TmaType;
template <> struct TmaType<float> { static constexpr CUtensorMapDataType v = CU_TENSOR_MAP_DATA_TYPE_FLOAT32; };
template <> struct TmaType<__half> { static constexpr CUtensorMapDataType v = CU_TENSOR_MAP_DATA_TYPE_FLOAT16; };
template <> struct TmaType<__nv_bfloat16> { static constexpr CUtensorMapDataType v = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16; };

static int log2_of(int64_t v) {
    int s = 0;
    while ((int64_t(1) << s) < v) ++s;
    return s;
}

template <typename T, int BITS, bool PACK>
static int launch_rows_tma(const T* x, int64_t n_rows, int lanes_per_block, uint8_t* q, float* scale, float* zp,
                           cudaStream_t st) {
    using RL = RowLayout<T>;
    CUtensorMap tmap;
    int rc = make_tensor_map_2d(&tmap, TmaType<T>::v, sizeof(T), x, kRowElems, (uint64_t)n_rows, RL::kRowBytes,
                                kRowElems, kTileRows,
                                sizeof(T) == 4 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
    auto kern = quantize_rows_tma_kernel<T, BITS, PACK>;
    const int smem = kStages * RL::kTileBytes + 1024;
    if (int e = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), smem)) return e;
    const int64_t n_tiles = (n_rows + kTileRows - 1) / kTileRows;
    cudaError_t e = launch_pdl(kern, dim3((unsigned)n_tiles), dim3(kTmaThreads), (size_t)smem, st, tmap, n_rows,
                               log2_of(lanes_per_block), q, scale, zp);
    return cuda_status(e != cudaSuccess ? e : cudaGetLastError());
}

// One cooperative launch: a CTA per SM (or per tile when there are fewer tiles).
template <typename T, int BITS, bool PACK, int CONV>
static int launch_tensor_fused(const T* x, int64_t n, int64_t n_rows, uint8_t* q, float* scale, float* zp, float* ws,
                               cudaStream_t st) {
    using RL = RowLayout<T>;
    constexpr int kTileBytes = kFRows * RL::kRowBytes;
    CUtensorMap tmap;
    int rc = make_tensor_map_2d(&tmap, TmaType<T>::v, sizeof(T), x, kRowElems, (uint64_t)n_rows, RL::kRowBytes,
                                kRowElems, kFRows,
                                sizeof(T) == 4 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
    auto kern = quantize_tensor_fused_kernel<T, BITS, PACK, CONV>;
    int nslots = (224 * 1024) / kTileBytes;                      // 14 x 16 KB (+1 KB alignment) of the 227 KB an SM offers
    if (nslots > kFMaxSlots) nslots = kFMaxSlots;
    int ring_min = (128 * 1024) / kTileBytes;                    // 128 KB in flight per SM (a stage is held until its loads have returned)
    ring_min = (ring_min + kFGroups - 1) / kFGroups * kFGroups;
    const int smem = nslots * kTileBytes + 1024;
    if (int e = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), smem)) return e;
    const int64_t n_tiles = (n_rows + kFRows - 1) / kFRows;
    cudaLaunchConfig_t cfg = {};
    const int sms = device_sm_count();
    cfg.gridDim = dim3((unsigned)(n_tiles < sms ? n_tiles : sms));
    cfg.blockDim = dim3(kFThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;                 // the grid barrier needs every CTA resident
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cuda_status(cudaLaunchKernelEx(&cfg, kern, tmap, x, n, n_rows, nslots, ring_min, q, scale, zp, ws));
}

static bool is_pow2(int64_t v) { return v > 0 && (v & (v - 1)) == 0; }
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// DIM0, convention A: one cooperative launch when the matrix tiles cleanly; returns -1 when the
// shape is not eligible (the caller falls back to the multi-launch path).
template <typename T, int BITS, bool PACK>
static int launch_dim0_fused(const T* x, int64_t rows, int64_t cols, uint8_t* q, float* scale, float* zp, float* ws,
                             cudaStream_t st) {
    using RL = RowLayout<T>;
    constexpr int kTileBytes = kFRows * RL::kRowBytes;
    if (cols % kRowElems != 0 || !aligned16(x) || !aligned16(q)) return -1;
    // the second pass lives on L2 hits: beyond ~100 MB the re-read comes from HBM anyway and the
    // multi-launch path (more CTAs in flight) measured faster
    if ((double)rows * (double)cols * sizeof(T) > 100e6) return -1;
    Dim0Geom geo;
    const int64_t tps = (rows + kFRows - 1) / kFRows, n_strips = cols / kRowElems;
    if (tps * n_strips > (int64_t)1 << 30) return -1;
    geo.tps = (int)tps;
    geo.n_tiles = (int)(tps * n_strips);
    const int sms = device_sm_count();
    const int G = geo.n_tiles < sms ? geo.n_tiles : sms;
    const int per_cta = (geo.n_tiles + G - 1) / G;
    geo.max_strips = (per_cta + geo.tps - 1) / geo.tps + 1;
    if (geo.max_strips > kD0MaxStrips) return -1;
    CUtensorMap tmap;
    int rc = make_tensor_map_2d(&tmap, TmaType<T>::v, sizeof(T), x, (uint64_t)cols, (uint64_t)rows,
                                (uint64_t)cols * sizeof(T), kRowElems, kFRows,
                                sizeof(T) == 4 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
    auto kern = quantize_dim0_fused_kernel<T, BITS, PACK>;
    int nslots = (192 * 1024) / kTileBytes;                      // 12 x 16 KB; staging (16 KB) and the parameter tables (10 KB) take the rest
    if (nslots > kFMaxSlots) nslots = kFMaxSlots;
    int ring_min = (64 * 1024) / kTileBytes;
    ring_min = (ring_min + kFGroups - 1) / kFGroups * kFGroups;
    const int smem = nslots * kTileBytes + kFGroups * kFRows * 32 + 1024;      // + one staging tile per group
    if (int e = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), smem)) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)G);
    cfg.blockDim = dim3(kFThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cuda_status(cudaLaunchKernelEx(&cfg, kern, tmap, rows, cols, geo, nslots, ring_min, q, scale, zp, ws));
}


// TENSOR / DIM0 body shared by conventions A and B.
template <typename T, int BITS, bool PACK, int CONV>
static int quantize_reduced(const T* x, int64_t rows, int64_t cols, int mode, uint8_t* q, float* scale, float* zp,
                            float* ws, cudaStream_t st) {
    const int64_t n = rows * cols;
    if (mode == QUANTA_MODE_TENSOR) {
        const int64_t n_rows = aligned16(x) && aligned16(q) ? n / kRowElems : 0;
        int64_t start = 0;
        if (n_rows > 0) {
            int rc = launch_tensor_fused<T, BITS, PACK, CONV>(x, n, n_rows, q, scale, zp, ws, st);
            if (rc) return rc;
            start = n_rows * kRowElems;
        } else {
            // unaligned pointers (or fewer than kRowElems elements): partial min/max, finalize, generic quantize
            float* pmin = ws + kWsHeaderFloats + 64;
            float* pmax = pmin + kMaxPartialCtas;
            int64_t want = (n + 256 * 16 - 1) / (256 * 16);
            const int cap = kNumSMs * 4;                       // 4 resident CTAs of 256 threads per SM
            int g = (int)(want < 1 ? 1 : (want > cap ? cap : want));
            launch_pdl(minmax_tensor_partial_kernel<T>, g, dim3(256), 0, st, x, n, pmin, pmax);
            launch_pdl(minmax_tensor_finalize_kernel<CONV>, dim3(1), dim3(256), 0, st, pmin, pmax, g, BITS, scale, zp, ws);
        }
        if (start < n) {
            int64_t pairs = (n - start + 1) / 2;
            launch_pdl(quantize_generic_kernel<T, BITS, PACK, CONV>, dim3((unsigned)((pairs + 255) / 256)), dim3(256), 0, st, 
                x, start, n, 1, q, scale, zp, ws);
        }
        return cuda_status(cudaGetLastError());
    }
    // DIM0
    if (CONV == kConvA) {
        const int rc = launch_dim0_fused<T, BITS, PACK>(x, rows, cols, q, scale, zp, ws, st);
        if (rc >= 0) return rc;
    }
    float* rcp = ws + kWsHeaderFloats;
    float* pmin = rcp + cols;
    int nchunks = (int)((rows + 63) / 64);
    if (nchunks > kMaxDim0Chunks) nchunks = kMaxDim0Chunks;
    if (nchunks < 1) nchunks = 1;
    const int rpc = (int)((rows + nchunks - 1) / nchunks);
    nchunks = (int)((rows + rpc - 1) / rpc);
    float* pmax = pmin + (int64_t)nchunks * cols;
    const bool fast = (cols % 4 == 0) && aligned16(x) && aligned16(q) && aligned16(ws);
    if (CONV != kConvA) launch_pdl(dim0_flag_init_kernel, dim3(1), dim3(1), 0, st, ws, 1);
    if (fast) {
        dim3 g((unsigned)((cols / 4 + 127) / 128), nchunks);
        launch_pdl(minmax_dim0_partial_kernel<T>, g, dim3(128), 0, st, x, rows, cols, rpc, pmin, pmax);
    } else {
        dim3 g((unsigned)((cols + 127) / 128), nchunks);
        launch_pdl(minmax_dim0_partial_generic_kernel<T>, g, dim3(128), 0, st, x, rows, cols, rpc, pmin, pmax);
    }
    launch_pdl(minmax_dim0_finalize_kernel<CONV>, dim3((unsigned)((cols + 31) / 32)), dim3(32), 0, st, pmin, pmax, nchunks, cols, BITS,
                                                                                  scale, zp, ws);
    if (CONV != kConvA) launch_pdl(dim0_earlyout_params_kernel, dim3((unsigned)((cols + 127) / 128)), dim3(128), 0, st, cols, scale, zp, ws);
    if (fast) {
        int qchunks = (int)((rows + 31) / 32);
        if (qchunks > 1024) qchunks = 1024;
        const int qrpc = (int)((rows + qchunks - 1) / qchunks);
        qchunks = (int)((rows + qrpc - 1) / qrpc);
        dim3 g((unsigned)((cols / 4 + 127) / 128), qchunks);
        launch_pdl(quantize_dim0_kernel<T, BITS, PACK, CONV>, g, dim3(128), 0, st, x, rows, cols, qrpc, q, scale, zp, ws);
    } else {
        int64_t pairs = (n + 1) / 2;
        launch_pdl(quantize_generic_kernel<T, BITS, PACK, CONV>, dim3((unsigned)((pairs + 255) / 256)), dim3(256), 0, st, 
            x, 0, n, cols, q, scale, zp, ws);
    }
    return cuda_status(cudaGetLastError());
}

template <typename T, int BITS, bool PACK>
static int quantize_affine_t(const T* x, int64_t rows, int64_t cols, int mode, int64_t block, uint8_t* q, float* scale,
                             float* zp, float* ws, cudaStream_t st) {
    const int64_t n = rows * cols;
    if (mode == QUANTA_MODE_BLOCK) {
        const int64_t nblocks = n / block;
        if (block % kRowElems == 0 && is_pow2(block / kRowElems) && block <= 1024 && aligned16(x) && aligned16(q))
            return launch_rows_tma<T, BITS, PACK>(x, n / kRowElems, (int)(block / kRowElems), q, scale, zp, st);
        if (PACK && (block & 1)) return QUANTA_EUNSUPPORTED;
        launch_pdl(quantize_block_generic_kernel<T, BITS, PACK>, dim3((unsigned)((nblocks + 7) / 8)), dim3(256), 0, st, x, nblocks, block, q,
                                                                                                  scale, zp);
        return cuda_status(cudaGetLastError());
    }
    return quantize_reduced<T, BITS, PACK, kConvA>(x, rows, cols, mode, q, scale, zp, ws, st);
}

template <typename T>
static int quantize_affine_bits(const T* x, int64_t rows, int64_t cols, int mode, int64_t block, int bits, int pack,
                                uint8_t* q, float* scale, float* zp, float* ws, cudaStream_t st) {
    if (bits == 8) return quantize_affine_t<T, 8, false>(x, rows, cols, mode, block, q, scale, zp, ws, st);
    if (pack) return quantize_affine_t<T, 4, true>(x, rows, cols, mode, block, q, scale, zp, ws, st);
    return quantize_affine_t<T, 4, false>(x, rows, cols, mode, block, q, scale, zp, ws, st);
}

template <typename T>
static int backend_quantize_t(const T* x, int64_t rows, int64_t cols, int per_channel, int symmetric, int bits,
                              uint8_t* q, float* scale, float* zp, float* ws, cudaStream_t st) {
    const int mode = per_channel ? QUANTA_MODE_DIM0 : QUANTA_MODE_TENSOR;
    if (bits == 8) {
        return symmetric ? quantize_reduced<T, 8, false, kConvBSym>(x, rows, cols, mode, q, scale, zp, ws, st)
                         : quantize_reduced<T, 8, false, kConvBAsym>(x, rows, cols, mode, q, scale, zp, ws, st);
    }
    return symmetric ? quantize_reduced<T, 4, false, kConvBSym>(x, rows, cols, mode, q, scale, zp, ws, st)
                     : quantize_reduced<T, 4, false, kConvBAsym>(x, rows, cols, mode, q, scale, zp, ws, st);
}

// Blockwise batch: tensors that qualify for the TMA stream go through the multi-tensor kernel in
// groups of kMultiMax; anything else falls back to a per-tensor launch.  Consecutive multi-tensor
// launches overlap: each releases the next early (kReleaseNext), which then waits before it exits
// instead of before it starts; a per-tensor launch in between, and the end of the call, break the chain.
template <typename T, int BITS, bool PACK>
static int quantize_block_batch_t(const void* const* xs, const int64_t* numels, int count, int64_t block,
                                  uint8_t* const* qs, float* const* scales, float* const* zps, cudaStream_t st) {
    using RL = RowLayout<T>;
    const bool shape_ok = block % kRowElems == 0 && is_pow2(block / kRowElems) && block <= 1024;
    auto kern = quantize_rows_tma_multi_kernel<T, BITS, PACK>;
    const int smem = kStages * RL::kTileBytes + 1024;
    if (int e = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), smem)) return e;
    MultiArgs args;
    args.count = 0;
    args.tile_base[0] = 0;
    bool released = false;                 // the previous launch on `st` is a multi-tensor launch that released us
    auto flush = [&](bool release_next) -> int {
        if (args.count == 0) return QUANTA_OK;
        const int pdl = (released ? 0 : kWaitFirst) | (release_next ? kReleaseNext : 0);
        cudaError_t le = launch_pdl(kern, dim3((unsigned)args.tile_base[args.count]), dim3(kTmaThreads), (size_t)smem, st, args,
                                    log2_of(block / kRowElems), pdl);
        if (le != cudaSuccess) return (int)le;
        released = release_next;
        args.count = 0;
        args.tile_base[0] = 0;
        return cuda_status(cudaGetLastError());
    };
    // A launch that released the next one must be followed by it: otherwise the next programmatic launch on the
    // stream could start before the released launch completes.  So an input error after a release still launches the
    // pending group (which waits for its predecessor before it exits) before it is returned.  Only a failing launch
    // can leave a released launch without its successor; the call returns that launch error.
    auto fail = [&](int rc) -> int {
        if (released) flush(false);
        return rc;
    };
    for (int i = 0; i < count; ++i) {
        const T* x = static_cast<const T*>(xs[i]);
        const int64_t n = numels[i];
        if (n <= 0 || n % block != 0) return fail(QUANTA_EINVAL);
        const int64_t n_rows = n / kRowElems;
        const int64_t tiles = (n_rows + kTileRows - 1) / kTileRows;
        if (!shape_ok || !aligned16(x) || !aligned16(qs[i]) || tiles > (int64_t)1 << 24) {
            int rc = flush(false);
            if (rc) return rc;
            rc = quantize_affine_t<T, BITS, PACK>(x, 1, n, QUANTA_MODE_BLOCK, block, qs[i], scales[i], zps[i], nullptr, st);
            if (rc) return rc;
            continue;
        }
        // encoded before a flush that releases the next launch, so that a releasing flush always has a group to follow it
        CUtensorMap map;
        int rc = make_tensor_map_2d(&map, TmaType<T>::v, sizeof(T), x, kRowElems, (uint64_t)n_rows, RL::kRowBytes,
                                    kRowElems, kTileRows,
                                    sizeof(T) == 4 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B);
        if (rc) return fail(rc);
        if (args.count == kMultiMax || (int64_t)args.tile_base[args.count] + tiles > (int64_t)1 << 30) {
            rc = flush(true);
            if (rc) return rc;
        }
        const int k = args.count;
        args.maps[k] = map;
        args.n_rows[k] = n_rows;
        args.q[k] = qs[i]; args.scale[k] = scales[i]; args.zp[k] = zps[i];
        args.tile_base[k + 1] = args.tile_base[k] + (int)tiles;
        args.count = k + 1;
    }
    return flush(false);
}

size_t quantize_workspace_bytes(int64_t cols) {
    size_t tensor_part = (size_t)(kWsHeaderFloats + 64 + 2 * kMaxPartialCtas) * 4;
    // multi-launch path: rcp + chunk partials; single-launch path: cols + (cols/32 + 3 * #SMs) partial slots of 64
    size_t dim0_part = (size_t)(kWsHeaderFloats + (int64_t)(2 * kMaxDim0Chunks + 1) * (cols < 1 ? 1 : cols) +
                                4 * kNumSMs * kD0SlotFloats + 64) * 4;
    return (tensor_part > dim0_part ? tensor_part : dim0_part) + 256;
}

}  // namespace quanta

using namespace quanta;

extern "C" int quanta_quantize_affine(const void* x, int x_dtype, int64_t rows, int64_t cols, int mode, int64_t block,
                                      int bits, int pack4, uint8_t* q_out, float* scale_out, float* zp_out,
                                      void* workspace, size_t workspace_bytes, void* stream) {
    if (!x || !q_out || !scale_out || !zp_out) return QUANTA_EINVAL;
    if (rows <= 0 || cols <= 0 || (bits != 8 && bits != 4) || (pack4 && bits != 4)) return QUANTA_EINVAL;
    if (mode < QUANTA_MODE_TENSOR || mode > QUANTA_MODE_BLOCK) return QUANTA_EINVAL;
    if (mode == QUANTA_MODE_BLOCK && (block <= 0 || (rows * cols) % block != 0)) return QUANTA_EINVAL;
    if (mode != QUANTA_MODE_BLOCK) {
        if (!workspace) return QUANTA_EINVAL;
        if (workspace_bytes < quantize_workspace_bytes(mode == QUANTA_MODE_DIM0 ? cols : 1)) return QUANTA_EWORKSPACE;
    }
    float* ws = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (x_dtype) {
        case QUANTA_F32:
            return quantize_affine_bits(static_cast<const float*>(x), rows, cols, mode, block, bits, pack4, q_out,
                                        scale_out, zp_out, ws, st);
        case QUANTA_F16:
            return quantize_affine_bits(static_cast<const __half*>(x), rows, cols, mode, block, bits, pack4, q_out,
                                        scale_out, zp_out, ws, st);
        case QUANTA_BF16:
            return quantize_affine_bits(static_cast<const __nv_bfloat16*>(x), rows, cols, mode, block, bits, pack4,
                                        q_out, scale_out, zp_out, ws, st);
    }
    return QUANTA_EINVAL;
}

extern "C" int quanta_backend_quantize(const void* x, int x_dtype, int64_t rows, int64_t cols, int per_channel,
                                       int symmetric, int bits, uint8_t* q_out, float* scale_out, float* zp_out,
                                       void* workspace, size_t workspace_bytes, void* stream) {
    if (!x || !q_out || !scale_out || !zp_out || !workspace) return QUANTA_EINVAL;
    if (rows <= 0 || cols <= 0 || (bits != 8 && bits != 4)) return QUANTA_EINVAL;
    if (workspace_bytes < quantize_workspace_bytes(per_channel ? cols : 1)) return QUANTA_EWORKSPACE;
    float* ws = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (x_dtype) {
        case QUANTA_F32:
            return backend_quantize_t(static_cast<const float*>(x), rows, cols, per_channel, symmetric, bits, q_out,
                                      scale_out, zp_out, ws, st);
        case QUANTA_F16:
            return backend_quantize_t(static_cast<const __half*>(x), rows, cols, per_channel, symmetric, bits, q_out,
                                      scale_out, zp_out, ws, st);
        case QUANTA_BF16:
            return backend_quantize_t(static_cast<const __nv_bfloat16*>(x), rows, cols, per_channel, symmetric, bits,
                                      q_out, scale_out, zp_out, ws, st);
    }
    return QUANTA_EINVAL;
}

extern "C" int quanta_quantize_block_batch(const void* const* xs, const int64_t* numels, int count, int x_dtype,
                                           int64_t block, int bits, int pack4, uint8_t* const* q_outs,
                                           float* const* scale_outs, float* const* zp_outs, void* stream) {
    if (!xs || !numels || !q_outs || !scale_outs || !zp_outs || count < 0) return QUANTA_EINVAL;
    if ((bits != 8 && bits != 4) || (pack4 && bits != 4) || block <= 0) return QUANTA_EINVAL;
    for (int i = 0; i < count; ++i)
        if (!xs[i] || !q_outs[i] || !scale_outs[i] || !zp_outs[i]) return QUANTA_EINVAL;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
#define QUANTA_BATCH(T)                                                                                              \
    (bits == 8 ? quantize_block_batch_t<T, 8, false>(xs, numels, count, block, q_outs, scale_outs, zp_outs, st)      \
               : (pack4 ? quantize_block_batch_t<T, 4, true>(xs, numels, count, block, q_outs, scale_outs, zp_outs, st) \
                        : quantize_block_batch_t<T, 4, false>(xs, numels, count, block, q_outs, scale_outs, zp_outs, st)))
    switch (x_dtype) {
        case QUANTA_F32: return QUANTA_BATCH(float);
        case QUANTA_F16: return QUANTA_BATCH(__half);
        case QUANTA_BF16: return QUANTA_BATCH(__nv_bfloat16);
    }
#undef QUANTA_BATCH
    return QUANTA_EINVAL;
}
