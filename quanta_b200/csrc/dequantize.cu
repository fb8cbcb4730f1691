// Dequantize kernels (rows A4, B2 of SURVEY §8) and their C-ABI entry points.
//
// Output-bandwidth bound (1 B in, 4 B out per code).  Every warp store is a
// fully coalesced 512-byte STG.128 sweep; codes are widened with one PRMT into
// the mantissa of 2^23 (exact u8 -> fp32, no I2F), then the reference's two
// separately rounded operations are applied with explicit _rn intrinsics.
#include "common.cuh"

namespace quanta {

enum DqConv : int { kDqA = 0, kDqB = 1 };

// exact float(byte k of w)
template <int K>
__device__ __forceinline__ float byte_to_f32(uint32_t w) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(0x4B000000u), "r"(0x7540u + K));
    return __fsub_rn(__uint_as_float(r), 8388608.0f);
}

struct DqParam {
    float s, z;
    float rcp;      // conv B: RN(1/s) when the hoisted-reciprocal divide is exact, else 0
};

// conv B divides every element by the scale.  With y = RN(1/s) hoisted out of the element loop,
// q0 = a*y; r = fma(-s, q0, a); q = fma(y, r, q0) is the correctly rounded a/s for every integer
// |a| <= 510 and s in [2^-100, 2^100] (checked on the CPU over 4.3e9 pairs, 0 mismatches against
// the IEEE divide); codes minus an integer zero-point with |zp| <= 255 are such integers.
// Anything else takes the generic divide.
__device__ __forceinline__ float dq_rcp(float s, float z) {
    const float as = fabsf(s);
    const bool ok = as >= 7.888609052210118e-31f && as <= 1.2676506002282294e30f && fabsf(z) <= 255.0f && z == rintf(z);
    return ok ? __frcp_rn(s) : 0.0f;
}

// conv A: RN(RN(q*s) + z)            (functional/quantization.py:38,58)
// conv B: RN(RN(q' - z) / s), q' = int8(q) - OFF when `sym`   (backends/cpu/quantization.py:80-84)
template <int CONV>
__device__ __forceinline__ float dq_value(float qf, const DqParam& p, bool sym, float off) {
    if (CONV == kDqA) return __fadd_rn(__fmul_rn(qf, p.s), p.z);
    if (sym) {
        // ((q - OFF + 128) mod 256) - 128: the reference's int8 arithmetic wraps
        float v = qf - off;                    // exact small integers in [-128, 247]
        v = v > 127.0f ? v - 256.0f : v;
        qf = v;
    }
    const float a = __fsub_rn(qf, p.z);
    if (p.rcp != 0.0f) {
        const float q0 = __fmul_rn(a, p.rcp);
        return __fmaf_rn(p.rcp, __fmaf_rn(-p.s, q0, a), q0);
    }
    return __fdiv_rn(a, p.s);
}

template <typename OUT> __device__ __forceinline__ void store4(OUT* dst, float a, float b, float c, float d);
template <> __device__ __forceinline__ void store4<float>(float* dst, float a, float b, float c, float d) {
    __stcs(reinterpret_cast<float4*>(dst), make_float4(a, b, c, d));
}
template <> __device__ __forceinline__ void store4<__half>(__half* dst, float a, float b, float c, float d) {
    __half2 lo = __floats2half2_rn(a, b), hi = __floats2half2_rn(c, d);
    uint2 v; v.x = *reinterpret_cast<uint32_t*>(&lo); v.y = *reinterpret_cast<uint32_t*>(&hi);
    __stcs(reinterpret_cast<uint2*>(dst), v);
}
template <> __device__ __forceinline__ void store4<__nv_bfloat16>(__nv_bfloat16* dst, float a, float b, float c, float d) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
    uint2 v; v.x = *reinterpret_cast<uint32_t*>(&lo); v.y = *reinterpret_cast<uint32_t*>(&hi);
    __stcs(reinterpret_cast<uint2*>(dst), v);
}
template <typename OUT> __device__ __forceinline__ OUT from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// 4 codes starting at element i (i % 4 == 0) as one 32-bit word of bytes.
template <bool PACKED>
__device__ __forceinline__ uint32_t load_codes4(const uint8_t* q, int64_t i) {
    if (!PACKED) return __ldcs(reinterpret_cast<const unsigned int*>(q + i));
    uint32_t h = __ldcs(reinterpret_cast<const unsigned short*>(q + (i >> 1)));
    // [n0 n1 | n2 n3] nibbles -> bytes n0, n1, n2, n3
    return (h & 0x000Fu) | ((h & 0x00F0u) << 4) | ((h & 0x0F00u) << 8) | ((h & 0xF000u) << 12);
}

// TENSOR / BLOCK: flat sweep, 4 codes per thread per step, params per step.
template <typename OUT, bool PACKED, int CONV>
__global__ void __launch_bounds__(256) dequant_flat_kernel(const uint8_t* __restrict__ q, int64_t n4, int block_shift,
                                                           int64_t block, const float* __restrict__ scale,
                                                           const float* __restrict__ zp, OUT* __restrict__ out,
                                                           const int* __restrict__ flag, float off) {
    pdl_enter();
    const bool sym = CONV == kDqB && flag[0] != 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    // per-tensor parameters (block == 0) are fetched and prepared once
    DqParam p0{0.0f, 0.0f, 0.0f};
    if (block == 0) {
        p0.s = __ldg(scale); p0.z = __ldg(zp);
        if (CONV == kDqB) p0.rcp = dq_rcp(p0.s, p0.z);
    }
    auto emit = [&](int64_t g, uint32_t w, float ps, float pz) {
        const int64_t i = g * 4;
        DqParam p = p0;
        if (block != 0) {
            p.s = ps; p.z = pz;
            if (CONV == kDqB) p.rcp = dq_rcp(p.s, p.z);
        }
        store4<OUT>(out + i, dq_value<CONV>(byte_to_f32<0>(w), p, sym, off), dq_value<CONV>(byte_to_f32<1>(w), p, sym, off),
                    dq_value<CONV>(byte_to_f32<2>(w), p, sym, off), dq_value<CONV>(byte_to_f32<3>(w), p, sym, off));
    };
    auto pidx = [&](int64_t g) -> int64_t {
        const int64_t i = g * 4;
        return block == 0 ? 0 : (block_shift >= 0 ? (i >> block_shift) : (i / block));
    };
    // 4 codes per thread per step keep a warp's accesses contiguous; 4 steps are in flight per thread
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; g + 3 * stride < n4; g += 4 * stride) {
        uint32_t w[4]; float ps[4], pz[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            w[k] = load_codes4<PACKED>(q, (g + k * stride) * 4);
            ps[k] = pz[k] = 0.0f;
            if (block != 0) { const int64_t b = pidx(g + k * stride); ps[k] = __ldg(scale + b); pz[k] = __ldg(zp + b); }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) emit(g + k * stride, w[k], ps[k], pz[k]);
    }
    for (; g < n4; g += stride) {
        const int64_t b = pidx(g);
        emit(g, load_codes4<PACKED>(q, g * 4), block != 0 ? __ldg(scale + b) : 0.0f, block != 0 ? __ldg(zp + b) : 0.0f);
    }
}

// DIM0: thread owns 4 consecutive columns and walks down a chunk of rows.
template <typename OUT, bool PACKED, int CONV>
__global__ void __launch_bounds__(128) dequant_dim0_kernel(const uint8_t* __restrict__ q, int64_t rows, int64_t cols,
                                                           int rows_per_chunk, const float* __restrict__ scale,
                                                           const float* __restrict__ zp, OUT* __restrict__ out,
                                                           const int* __restrict__ flag, float off) {
    const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (c >= cols) return;
    const bool sym = CONV == kDqB && flag[0] != 0;
    DqParam p[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { p[j].s = scale[c + j]; p[j].z = zp[c + j]; p[j].rcp = CONV == kDqB ? dq_rcp(p[j].s, p[j].z) : 0.0f; }
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r1 = min(rows, r0 + rows_per_chunk);
    auto emit = [&](int64_t r, uint32_t w) {
        const int64_t i = r * cols + c;
        store4<OUT>(out + i, dq_value<CONV>(byte_to_f32<0>(w), p[0], sym, off), dq_value<CONV>(byte_to_f32<1>(w), p[1], sym, off),
                    dq_value<CONV>(byte_to_f32<2>(w), p[2], sym, off), dq_value<CONV>(byte_to_f32<3>(w), p[3], sym, off));
    };
    int64_t r = r0;
    for (; r + 3 < r1; r += 4) {                  // four rows' loads in flight
        uint32_t w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) w[k] = load_codes4<PACKED>(q, (r + k) * cols + c);
#pragma unroll
        for (int k = 0; k < 4; ++k) emit(r + k, w[k]);
    }
    for (; r < r1; ++r) emit(r, load_codes4<PACKED>(q, r * cols + c));
}

// Any shape / alignment: one element per thread.  chan(i) = 0 | i / block | i % cols.
template <typename OUT, bool PACKED, int CONV>
__global__ void __launch_bounds__(256) dequant_generic_kernel(const uint8_t* __restrict__ q, int64_t start, int64_t n,
                                                              int mode, int64_t p, const float* __restrict__ scale,
                                                              const float* __restrict__ zp, OUT* __restrict__ out,
                                                              const int* __restrict__ flag, float off) {
    const int64_t i = start + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const bool sym = CONV == kDqB && flag[0] != 0;
    uint32_t code = PACKED ? ((q[i >> 1] >> ((i & 1) * 4)) & 0xFu) : q[i];
    const int64_t ch = mode == QUANTA_MODE_TENSOR ? 0 : (mode == QUANTA_MODE_BLOCK ? i / p : i % p);
    DqParam pr{scale[ch], zp[ch], 0.0f};
    out[i] = from_f32<OUT>(dq_value<CONV>((float)code, pr, sym, off));
}

// B2's host-side `torch.allclose(zero_point, 0)` evaluated on the device:
// flag = all(|zp| <= 1e-8)  (NaN -> not close).
__global__ void __launch_bounds__(256) zp_allclose_zero_kernel(const float* __restrict__ zp, int64_t nchan, int* flag) {
    int ok = 1;
    for (int64_t i = threadIdx.x; i < nchan; i += blockDim.x) {
        float a = fabsf(zp[i]);
        ok &= (zp[i] == 0.0f) || (a <= 1e-8f);
    }
    ok = __syncthreads_and(ok);
    if (threadIdx.x == 0) flag[0] = ok;
}

static int shift_of(int64_t v) {
    if (v <= 0 || (v & (v - 1))) return -1;
    int s = 0;
    while ((int64_t(1) << s) < v) ++s;
    return s;
}

template <typename OUT, bool PACKED, int CONV>
static int dequant_launch(const uint8_t* q, int64_t rows, int64_t cols, int mode, int64_t block, const float* scale,
                          const float* zp, OUT* out, const int* flag, float off, cudaStream_t st) {
    const int64_t n = rows * cols;
    const uintptr_t qa = reinterpret_cast<uintptr_t>(q), oa = reinterpret_cast<uintptr_t>(out);
    const bool ptr_ok = (qa % (PACKED ? 2 : 4) == 0) && (oa % (4 * sizeof(OUT)) == 0);
    if (mode == QUANTA_MODE_DIM0 && ptr_ok && cols % 4 == 0) {
        int chunks = (int)((rows + 31) / 32);
        if (chunks > 2048) chunks = 2048;
        const int rpc = (int)((rows + chunks - 1) / chunks);
        chunks = (int)((rows + rpc - 1) / rpc);
        dim3 g((unsigned)((cols / 4 + 127) / 128), chunks);
        dequant_dim0_kernel<OUT, PACKED, CONV><<<g, 128, 0, st>>>(q, rows, cols, rpc, scale, zp, out, flag, off);
        return cuda_status(cudaGetLastError());
    }
    int64_t done = 0;
    if (mode != QUANTA_MODE_DIM0 && ptr_ok && (mode == QUANTA_MODE_TENSOR || block % 4 == 0)) {
        const int64_t n4 = n / 4;
        if (n4 > 0) {
            int64_t want = (n4 + 255) / 256;
            int64_t cap = (int64_t)kNumSMs * 8 * 4;
            cudaError_t e = launch_pdl(dequant_flat_kernel<OUT, PACKED, CONV>, dim3((unsigned)(want < cap ? want : cap)), dim3(256), 0, st,
                                       q, n4, shift_of(block), mode == QUANTA_MODE_TENSOR ? (int64_t)0 : block, scale, zp, out, flag, off);
            if (e != cudaSuccess) return (int)e;
        }
        done = n4 * 4;
    }
    if (done < n) {
        const int64_t rest = n - done;
        dequant_generic_kernel<OUT, PACKED, CONV><<<(unsigned)((rest + 255) / 256), 256, 0, st>>>(
            q, done, n, mode, mode == QUANTA_MODE_BLOCK ? block : cols, scale, zp, out, flag, off);
    }
    return cuda_status(cudaGetLastError());
}

// ---- many tensors, one launch (blockwise, convention A) ---------------------------------------------------
// Dequantizing every recorded tensor of a model — the reference calls QuantizationState.dequantize_tensor
// (Quanta/functional/state.py:246-281) once per tensor — as one grid: every matrix
// launched on its own pays ~4 us of ramp and drain on a 10-40 us stream.  The tensors' 4-code groups are cut into
// chunks of kDqChunk groups; the chunk index space is the concatenation of the tensors' chunks, a persistent grid
// walks it.  Descriptors ride in the kernel parameters.
constexpr int kDqMultiMax = 16;
constexpr int kDqChunk = 256 * 4;                  // groups of 4 codes per chunk: 4 steps of a 256-thread CTA
struct DqMultiArgs {
    const uint8_t* q[kDqMultiMax];
    const float* scale[kDqMultiMax];
    const float* zp[kDqMultiMax];
    void* out[kDqMultiMax];
    int64_t n4[kDqMultiMax];                       // groups of 4 codes
    int64_t chunk_base[kDqMultiMax + 1];           // first global chunk of tensor i; [count] = total
    int count;
};

template <typename OUT, bool PACKED>
__global__ void __launch_bounds__(256) dequant_flat_multi_kernel(const __grid_constant__ DqMultiArgs a, int block_shift,
                                                                 int64_t block) {
    pdl_enter();
    const int64_t total = a.chunk_base[a.count];
    int ti = 0;
    for (int64_t c = blockIdx.x; c < total; c += gridDim.x) {
        while (ti + 1 < a.count && c >= a.chunk_base[ti + 1]) ++ti;
        const uint8_t* __restrict__ q = a.q[ti];
        const float* __restrict__ scale = a.scale[ti];
        const float* __restrict__ zp = a.zp[ti];
        OUT* __restrict__ out = static_cast<OUT*>(a.out[ti]);
        const int64_t n4 = a.n4[ti];
        const int64_t g0 = (c - a.chunk_base[ti]) * kDqChunk + threadIdx.x;
        uint32_t w[4]; float ps[4], pz[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int64_t g = g0 + k * 256;
            w[k] = 0u; ps[k] = pz[k] = 0.0f;
            if (g < n4) {
                const int64_t i = g * 4;
                const int64_t b = block_shift >= 0 ? (i >> block_shift) : (i / block);
                w[k] = load_codes4<PACKED>(q, i);
                ps[k] = __ldg(scale + b); pz[k] = __ldg(zp + b);
            }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int64_t g = g0 + k * 256;
            if (g < n4) {
                const DqParam p{ps[k], pz[k], 0.0f};
                store4<OUT>(out + g * 4, dq_value<kDqA>(byte_to_f32<0>(w[k]), p, false, 0.f), dq_value<kDqA>(byte_to_f32<1>(w[k]), p, false, 0.f),
                            dq_value<kDqA>(byte_to_f32<2>(w[k]), p, false, 0.f), dq_value<kDqA>(byte_to_f32<3>(w[k]), p, false, 0.f));
            }
        }
    }
}

template <typename OUT, bool PACKED>
static int dequant_multi_launch(const uint8_t* const* qs, const int64_t* numels, int count, int64_t block, const float* const* scales,
                                const float* const* zps, void* const* outs, cudaStream_t st) {
    for (int first = 0; first < count; first += kDqMultiMax) {
        DqMultiArgs a;
        a.count = count - first < kDqMultiMax ? count - first : kDqMultiMax;
        a.chunk_base[0] = 0;
        for (int i = 0; i < a.count; ++i) {
            a.q[i] = qs[first + i]; a.scale[i] = scales[first + i]; a.zp[i] = zps[first + i]; a.out[i] = outs[first + i];
            a.n4[i] = numels[first + i] / 4;
            a.chunk_base[i + 1] = a.chunk_base[i] + (a.n4[i] + kDqChunk - 1) / kDqChunk;
        }
        for (int i = a.count; i < kDqMultiMax; ++i) { a.q[i] = nullptr; a.scale[i] = nullptr; a.zp[i] = nullptr; a.out[i] = nullptr; a.n4[i] = 0; a.chunk_base[i + 1] = a.chunk_base[a.count]; }
        const int64_t total = a.chunk_base[a.count];
        const int64_t cap = (int64_t)kNumSMs * 8;
        cudaError_t e = launch_pdl(dequant_flat_multi_kernel<OUT, PACKED>, dim3((unsigned)(total < cap ? total : cap)), dim3(256), 0, st,
                                   a, shift_of(block), block);
        if (e != cudaSuccess) return (int)e;
    }
    return cuda_status(cudaGetLastError());
}

template <bool PACKED, int CONV>
static int dequant_dtype(const uint8_t* q, int64_t rows, int64_t cols, int mode, int64_t block, const float* scale,
                         const float* zp, void* out, int out_dtype, const int* flag, float off, cudaStream_t st) {
    switch (out_dtype) {
        case QUANTA_F32:
            return dequant_launch<float, PACKED, CONV>(q, rows, cols, mode, block, scale, zp, static_cast<float*>(out), flag, off, st);
        case QUANTA_F16:
            return dequant_launch<__half, PACKED, CONV>(q, rows, cols, mode, block, scale, zp, static_cast<__half*>(out), flag, off, st);
        case QUANTA_BF16:
            return dequant_launch<__nv_bfloat16, PACKED, CONV>(q, rows, cols, mode, block, scale, zp,
                                                               static_cast<__nv_bfloat16*>(out), flag, off, st);
    }
    return QUANTA_EINVAL;
}

}  // namespace quanta

using namespace quanta;

extern "C" int quanta_dequantize_affine(const uint8_t* q, int packed4, int64_t rows, int64_t cols, int mode,
                                        int64_t block, const float* scale, const float* zp, void* out, int out_dtype,
                                        void* stream) {
    if (!q || !scale || !zp || !out || rows <= 0 || cols <= 0) return QUANTA_EINVAL;
    if (mode < QUANTA_MODE_TENSOR || mode > QUANTA_MODE_BLOCK) return QUANTA_EINVAL;
    if (mode == QUANTA_MODE_BLOCK && (block <= 0 || (rows * cols) % block != 0)) return QUANTA_EINVAL;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return packed4 ? dequant_dtype<true, kDqA>(q, rows, cols, mode, block, scale, zp, out, out_dtype, nullptr, 0.f, st)
                   : dequant_dtype<false, kDqA>(q, rows, cols, mode, block, scale, zp, out, out_dtype, nullptr, 0.f, st);
}

extern "C" int quanta_backend_dequantize(const uint8_t* q, int64_t rows, int64_t cols, int64_t nchan, int bits,
                                         const float* scale, const float* zp, float* out, void* workspace,
                                         size_t workspace_bytes, void* stream) {
    if (!q || !scale || !zp || !out || !workspace || rows <= 0 || cols <= 0) return QUANTA_EINVAL;
    if ((bits != 8 && bits != 4) || (nchan != 1 && nchan != cols)) return QUANTA_EINVAL;
    if (workspace_bytes < 256) return QUANTA_EWORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int* flag = reinterpret_cast<int*>((reinterpret_cast<uintptr_t>(workspace) + 15) & ~uintptr_t(15));
    zp_allclose_zero_kernel<<<1, 256, 0, st>>>(zp, nchan, flag);
    const int mode = nchan == 1 ? QUANTA_MODE_TENSOR : QUANTA_MODE_DIM0;
    return dequant_dtype<false, kDqB>(q, rows, cols, mode, 0, scale, zp, out, QUANTA_F32, flag, bits == 8 ? 128.f : 8.f, st);
}

// The per-parameter dequantize loop of a model in ceil(count / 16) launches: tensor i = numels[i] codes (packed4: two
// per byte), blockwise parameters scales[i] / zps[i] of numels[i] / block floats, output outs[i] (out_dtype).  Host
// arrays of device pointers.  Every numel must be a positive multiple of `block`, block % 4 == 0; code pointers
// 4-byte (2-byte when packed), outputs 16-byte (fp32) / 8-byte (16-bit) aligned.
extern "C" int quanta_dequantize_block_batch(const uint8_t* const* qs, const int64_t* numels, int count, int packed4,
                                             int64_t block, const float* const* scales, const float* const* zps,
                                             void* const* outs, int out_dtype, void* stream) {
    if (!qs || !numels || !scales || !zps || !outs || count < 0) return QUANTA_EINVAL;
    if (block <= 0 || block % 4 != 0) return QUANTA_EINVAL;
    if (out_dtype != QUANTA_F32 && out_dtype != QUANTA_F16 && out_dtype != QUANTA_BF16) return QUANTA_EINVAL;
    const size_t out_align = out_dtype == QUANTA_F32 ? 16 : 8;
    for (int i = 0; i < count; ++i) {
        if (!qs[i] || !scales[i] || !zps[i] || !outs[i] || numels[i] <= 0 || numels[i] % block != 0) return QUANTA_EINVAL;
        if (reinterpret_cast<uintptr_t>(qs[i]) % (packed4 ? 2 : 4) != 0 || reinterpret_cast<uintptr_t>(outs[i]) % out_align != 0) return QUANTA_EINVAL;
    }
    if (count == 0) return QUANTA_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (out_dtype) {
        case QUANTA_F32:
            return packed4 ? dequant_multi_launch<float, true>(qs, numels, count, block, scales, zps, outs, st)
                           : dequant_multi_launch<float, false>(qs, numels, count, block, scales, zps, outs, st);
        case QUANTA_F16:
            return packed4 ? dequant_multi_launch<__half, true>(qs, numels, count, block, scales, zps, outs, st)
                           : dequant_multi_launch<__half, false>(qs, numels, count, block, scales, zps, outs, st);
        default:
            return packed4 ? dequant_multi_launch<__nv_bfloat16, true>(qs, numels, count, block, scales, zps, outs, st)
                           : dequant_multi_launch<__nv_bfloat16, false>(qs, numels, count, block, scales, zps, outs, st);
    }
}
