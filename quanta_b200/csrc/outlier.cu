// LLM.int8()-style outlier-split matmul (row G3 of SURVEY §8) behind
// Linear8bitLt.threshold (Quanta/nn/linear.py:20,25 — stored, never used by the
// reference; semantics defined by oracle/oracle_np.py:int8_outlier_matmul).
//
//   J  = { j : max_i |x[i,j]| > threshold }                       outlier feature columns
//   cx[i] = rcp(absmax_i over non-outlier columns) * 127           (B1-symmetric arithmetic)
//   qx[i,k] = clamp(rint(x[i,k] * cx[i]), -127, 127), 0 for k in J
//   y[i,n] = float(sum_k qx[i,k] qw[n,k]) / (cx[i] * cw[n])        int8 x int8 -> int32 on the tensor cores
//          + sum_{j in J} x[i,j] * round_act(qw[n,j] / cw[n])      16-bit part, fp32 accumulate
//          + bias[n]
//
// Launches on the caller's stream:
//   1. outlier_colmax_kernel + outlier_columns_kernel   column abs-max of x, flags, ordered list J
//   2. outlier_rowquant_kernel  per-row abs-max over non-outlier columns, cx, int8 codes qx
//   3. int8_gemm_kernel         tcgen05.mma.kind::i8 (A = qw, B = qx, both TMA-fed, SWIZZLE_128B),
//                               int32 accumulators in TMEM; the epilogue rescales, adds the
//                               outlier columns on the CUDA cores and stores y
#include "common.cuh"

#include <type_traits>

namespace quanta {

constexpr int kOTileN = 128;      // output features per CTA (UMMA M)
constexpr int kOBlockK = 128;     // int8 K values per stage: one 128-byte swizzle atom
constexpr int kOThreads = 32 * 6; // warp 0 TMA, warp 1 MMA + TMEM, warps 2-5 epilogue
constexpr int kOMaxStages = 8;

template <typename T> __device__ __forceinline__ float ld_act(const T* p);
template <> __device__ __forceinline__ float ld_act<__half>(const __half* p) { return __half2float(*p); }
template <> __device__ __forceinline__ float ld_act<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <typename T> __device__ __forceinline__ float round_act(float v);
template <> __device__ __forceinline__ float round_act<__half>(float v) { return __half2float(__float2half_rn(v)); }
template <> __device__ __forceinline__ float round_act<__nv_bfloat16>(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
template <typename T> __device__ __forceinline__ T to_act(float v);
template <> __device__ __forceinline__ __half to_act<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 to_act<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// ---- 1. outlier columns ------------------------------------------------------
// 1a. column abs-max: thread = column (coalesced across the CTA), blockIdx.y = chunk of 64 rows;
//     non-negative floats order like their bit patterns, so the chunks merge with atomicMax.
template <typename ACT>
__global__ void __launch_bounds__(256) outlier_colmax_kernel(const ACT* __restrict__ x, int M, int K,
                                                             unsigned int* __restrict__ colmax) {
    const int c = blockIdx.x * 256 + threadIdx.x;
    if (c >= K) return;
    const int r0 = blockIdx.y * 64, r1 = min(M, r0 + 64);
    float mx = 0.0f;
#pragma unroll 8
    for (int i = r0; i < r1; ++i) mx = fmaxf(mx, fabsf(ld_act(x + (int64_t)i * K + c)));
    if (gridDim.y == 1) colmax[c] = __float_as_uint(mx);        // one chunk covers every row: no merge, no memset needed
    else atomicMax(colmax + c, __float_as_uint(mx));
}

// 1b. flags and the ordered list J: one CTA, thread = a contiguous run of columns, ONE block-wide
//     exclusive scan of the per-thread counts (two barriers in all, whatever K is).
__global__ void __launch_bounds__(1024) outlier_columns_kernel(const unsigned int* __restrict__ colmax, int K, float threshold,
                                                               uint8_t* __restrict__ flag, int* __restrict__ jlist,
                                                               int* __restrict__ jcount) {
    __shared__ int warp_counts[32];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int c_per = (K + 1023) / 1024;
    const int c0 = tid * c_per, c1 = min(K, c0 + c_per);
    int cnt = 0;
    for (int c = c0; c < c1; ++c) {
        const int f = __uint_as_float(colmax[c]) > threshold ? 1 : 0;
        flag[c] = (uint8_t)f;
        cnt += f;
    }
    int incl = cnt;                                      // inclusive scan inside the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += up;
    }
    if (lane == 31) warp_counts[w] = incl;
    __syncthreads();
    int base = incl - cnt;
    for (int k = 0; k < w; ++k) base += warp_counts[k];
    if (cnt) {
        for (int c = c0; c < c1; ++c) if (__uint_as_float(colmax[c]) > threshold) jlist[base++] = c;
    }
    if (tid == 1023) *jcount = base;
}

// ---- 2. per-row int8 codes of the non-outlier part ----------------------------
template <typename ACT>
__global__ void __launch_bounds__(256) outlier_rowquant_kernel(const ACT* __restrict__ x, int K,
                                                               const uint8_t* __restrict__ flag,
                                                               float* __restrict__ cx, int8_t* __restrict__ qx) {
    const int i = blockIdx.x;
    const ACT* xr = x + (int64_t)i * K;
    float am = 0.0f;
    for (int k = threadIdx.x; k < K; k += 256) if (!flag[k]) am = fmaxf(am, fabsf(ld_act(xr + k)));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) am = fmaxf(am, __shfl_xor_sync(0xffffffffu, am, o));
    __shared__ float red[8];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = am;
    __syncthreads();
#pragma unroll
    for (int w = 0; w < 8; ++w) am = fmaxf(am, red[w]);
    // backends/cpu/quantization.py:44-47: scale = 127 / absmax == reciprocal(absmax) * 127
    const float c = am == 0.0f ? 1.0f : __fmul_rn(__frcp_rn(am), 127.0f);
    if (threadIdx.x == 0) cx[i] = c;
    int8_t* qr = qx + (int64_t)i * K;
    for (int k = threadIdx.x; k < K; k += 256) {
        float v = flag[k] ? 0.0f : __fmul_rn(ld_act(xr + k), c);
        v = fminf(fmaxf(rintf(v), -127.0f), 127.0f);
        qr[k] = (int8_t)(int)v;
    }
}

// 2'. the same with 8 columns per thread per step (16-byte activation loads, 8-byte flag loads and code
//     stores); needs K % 8 == 0 and 16-byte aligned rows.
template <typename ACT>
__global__ void __launch_bounds__(256) outlier_rowquant_vec_kernel(const ACT* __restrict__ x, int K,
                                                                   const uint8_t* __restrict__ flag,
                                                                   float* __restrict__ cx, int8_t* __restrict__ qx) {
    const int i = blockIdx.x;
    const ACT* xr = x + (int64_t)i * K;
    const int nvec = K >> 3;
    float am = 0.0f;
    for (int v = threadIdx.x; v < nvec; v += 256) {
        const uint4 d = __ldg(reinterpret_cast<const uint4*>(xr) + v);
        const uint2 f = __ldg(reinterpret_cast<const uint2*>(flag) + v);
        const ACT* e = reinterpret_cast<const ACT*>(&d);
        const uint8_t* fb = reinterpret_cast<const uint8_t*>(&f);
#pragma unroll
        for (int k = 0; k < 8; ++k) if (!fb[k]) am = fmaxf(am, fabsf(ld_act(e + k)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) am = fmaxf(am, __shfl_xor_sync(0xffffffffu, am, o));
    __shared__ float red[8];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = am;
    __syncthreads();
#pragma unroll
    for (int w = 0; w < 8; ++w) am = fmaxf(am, red[w]);
    const float c = am == 0.0f ? 1.0f : __fmul_rn(__frcp_rn(am), 127.0f);
    if (threadIdx.x == 0) cx[i] = c;
    int8_t* qr = qx + (int64_t)i * K;
    for (int v = threadIdx.x; v < nvec; v += 256) {
        const uint4 d = __ldg(reinterpret_cast<const uint4*>(xr) + v);
        const uint2 f = __ldg(reinterpret_cast<const uint2*>(flag) + v);
        const ACT* e = reinterpret_cast<const ACT*>(&d);
        const uint8_t* fb = reinterpret_cast<const uint8_t*>(&f);
        uint32_t packed[2] = {0u, 0u};
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            float t = fb[k] ? 0.0f : __fmul_rn(ld_act(e + k), c);
            t = fminf(fmaxf(rintf(t), -127.0f), 127.0f);
            packed[k >> 2] |= ((uint32_t)(int)t & 0xFFu) << (8 * (k & 3));
        }
        *(reinterpret_cast<uint2*>(qr) + v) = make_uint2(packed[0], packed[1]);
    }
}

// ---- 3. int8 x int8 -> int32 GEMM + epilogue ------------------------------------
__device__ __forceinline__ void tma_load_2d_o(uint32_t dst, const CUtensorMap* map, uint32_t bar, int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ uint64_t desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ bool elect_one_o() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(pred));
    return pred != 0;
}

struct OutlierParams {
    int M, N, K;
    int mb;           // UMMA N: batch rows per CTA (multiple of 16, <= 256)
    int stages;
    int tmem_cols;
    int y_tma;        // y leaves through shared-memory staging + TMA stores (pointer / pitch aligned)
    int splits;       // K is cut into `splits` ranges (gridDim.z); int32 partial sums meet in `acc` (exact, order-free)
    uint32_t a_bytes, b_bytes;
};
constexpr int kOJ = 32;           // outlier columns handled per pass of the epilogue
constexpr uint32_t kOEpiBytes = 2 * 16 * 128 * 2 + kOJ * 256 * 4 + kOJ * 128 * 4 + 256 * 4;

template <typename ACT>
__global__ void __launch_bounds__(kOThreads, 1)
int8_gemm_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_x,
                 const __grid_constant__ CUtensorMap tmap_y, const ACT* __restrict__ x, const int8_t* __restrict__ qw, const float* __restrict__ cw,
                 const float* __restrict__ cx, const int* __restrict__ jlist, const int* __restrict__ jcount,
                 const ACT* __restrict__ bias, ACT* __restrict__ y, int* __restrict__ acc,
                 unsigned int* __restrict__ tile_counters, const __grid_constant__ OutlierParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t full[kOMaxStages], empty[kOMaxStages], d_full;
    __shared__ uint32_t tmem_slot;
    // epilogue tables, carved from dynamic shared memory behind the operand ring (kOEpiBytes):
    //   ystage[2][16][128] 16-bit (TMA-store staging) | xo[kOJ][256] | wos[kOJ][128] | cxs[256]
    const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int n0 = blockIdx.x * kOTileN, m0 = blockIdx.y * p.mb;
    const int nk_all = (p.K + kOBlockK - 1) / kOBlockK;
    // split-K: this CTA's range of 128-K blocks
    const int kb_lo = (int)((int64_t)nk_all * blockIdx.z / p.splits), kb_hi = (int)((int64_t)nk_all * (blockIdx.z + 1) / p.splits);
    const int nk = kb_hi - kb_lo;
    const uint32_t stage_bytes = p.a_bytes + p.b_bytes;
    __shared__ int last_flag;
    uint8_t* epi = smem_raw + (smem - smem_u32(smem_raw)) + (size_t)p.stages * stage_bytes;       // 1 KB aligned
    uint16_t (*ystage)[16][kOTileN] = reinterpret_cast<uint16_t (*)[16][kOTileN]>(epi);
    float (*xo)[256] = reinterpret_cast<float (*)[256]>(epi + 2 * 16 * kOTileN * 2);             // x[m0 + m, J[t]]
    float (*wos)[kOTileN] = reinterpret_cast<float (*)[kOTileN]>(epi + 2 * 16 * kOTileN * 2 + kOJ * 256 * 4);   // round_act(qw[n, J[t]] / cw[n])
    float* cxs = reinterpret_cast<float*>(epi + 2 * 16 * kOTileN * 2 + kOJ * 256 * 4 + kOJ * kOTileN * 4);      // cx[m0 + m]

    if (tid == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(&d_full, 1);
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_slot;

    if (warp == 0) {
        // ===== TMA producer: weight codes [128 x 128 B] and activation codes [mb x 128 B] per stage =====
        if (lane == 0) { prefetch_tensormap(&tmap_w); prefetch_tensormap(&tmap_x); }
        int s = 0;
        uint32_t ph = 0;
        for (int kb = 0; kb < nk; ++kb) {
            mbar_wait(&empty[s], ph ^ 1);
            if (elect_one_o()) {
                mbar_arrive_expect_tx(&full[s], stage_bytes);
                const uint32_t dst = smem + (uint32_t)s * stage_bytes;
                tma_load_2d_o(dst, &tmap_w, smem_u32(&full[s]), (kb_lo + kb) * kOBlockK, n0);
                tma_load_2d_o(dst + p.a_bytes, &tmap_x, smem_u32(&full[s]), (kb_lo + kb) * kOBlockK, m0);
            }
            __syncwarp();
            if (++s == p.stages) { s = 0; ph ^= 1; }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: 4 x (K = 32) tcgen05.mma.kind::i8 per stage =====
        // instruction descriptor: D = S32, A = B = signed int8, K-major, N = mb, M = 128
        const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.mb >> 3) << 17) | ((uint32_t)(kOTileN >> 4) << 24);
        int s = 0;
        uint32_t ph = 0;
        for (int kb = 0; kb < nk; ++kb) {
            mbar_wait(&full[s], ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (elect_one_o()) {
                const uint64_t da = desc_sw128(smem + (uint32_t)s * stage_bytes);
                const uint64_t db = desc_sw128(smem + (uint32_t)s * stage_bytes + p.a_bytes);
#pragma unroll
                for (int k = 0; k < kOBlockK / 32; ++k) {
                    const uint32_t acc = (kb != 0 || k != 0) ? 1u : 0u;
                    asm volatile(
                        "{\n\t"
                        ".reg .pred p;\n\t"
                        "setp.ne.b32 p, %4, 0;\n\t"
                        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
                        "}\n" ::"r"(tmem), "l"(da + 2 * k), "l"(db + 2 * k), "r"(idesc), "r"(acc) : "memory");
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&empty[s])) : "memory");
                if (kb == nk - 1)
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&d_full)) : "memory");
            }
            __syncwarp();
            if (++s == p.stages) { s = 0; ph ^= 1; }
        }
    } else {
        // ===== epilogue: TMEM lane = output feature =====
        const int quarter = warp & 3;
        const int row = 32 * quarter + lane;
        const int etid = tid - 64;                                  // 0..127 over the 4 epilogue warps
        const int gn = n0 + row;
        const bool n_ok = gn < p.N;
        const float cwn = n_ok ? cw[gn] : 1.0f;
        const float b = (bias != nullptr && n_ok) ? ld_act(bias + gn) : 0.0f;
        const int nj = *jcount;
        const int8_t* qrow = qw + (int64_t)(n_ok ? gn : 0) * p.K;
        const int m_valid = min(p.mb, p.M - m0);
        if (etid == 0 && p.y_tma) prefetch_tensormap(&tmap_y);
        // while the main loop runs: this tile's row multipliers and the first pass of outlier operands
        for (int m = etid; m < p.mb; m += 128) cxs[m] = m < m_valid ? cx[m0 + m] : 1.0f;
        auto stage_outliers = [&](int t0) {
            const int nt = min(kOJ, nj - t0);
            for (int t = 0; t < nt; ++t) {
                const int jc = jlist[t0 + t];
                // x[m, j] * round_act(qw[n, j] / cw[n]): the weight factor of this thread's feature
                wos[t][row] = round_act<ACT>(__fdiv_rn((float)qrow[jc], cwn));
                for (int m = etid; m < p.mb; m += 128) xo[t][m] = m < m_valid ? ld_act(x + (int64_t)(m0 + m) * p.K + jc) : 0.0f;
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
        };
        const bool single_pass = nj <= kOJ;
        if (single_pass) stage_outliers(0); else asm volatile("bar.sync 1, 128;" ::: "memory");      // cxs visible
        mbar_wait(&d_full, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t taddr = tmem + ((uint32_t)(32 * quarter) << 16);
        bool from_acc = false;
        if (p.splits > 1) {
            // int32 partial sums are exact, so the K ranges may meet in any order: add this range into the
            // (zero-initialised) accumulator, then the CTA that arrives last at the tile's counter finishes the tile
            for (int c0 = 0; c0 < m_valid; c0 += 16) {
                uint32_t r[16];
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                      "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                    : "r"(taddr + c0) : "memory");
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (n_ok) {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (c0 + j < m_valid) atomicAdd(acc + (int64_t)(m0 + c0 + j) * p.N + gn, (int)r[j]);
                }
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (etid == 0) {
                __threadfence();
                const unsigned int old = atomicAdd(tile_counters + blockIdx.y * gridDim.x + blockIdx.x, 1u);
                __threadfence();
                last_flag = (old == (unsigned int)(p.splits - 1)) ? 1 : 0;
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            from_acc = true;
        }
        if (from_acc && !last_flag) {
            // not the last range of this tile: nothing more to do
        } else
        for (int c0 = 0; c0 < p.mb; c0 += 16) {
            uint32_t r[16];
            if (!from_acc) {
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                      "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                    : "r"(taddr + c0) : "memory");
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    r[j] = (n_ok && c0 + j < m_valid) ? (uint32_t)__ldcg(acc + (int64_t)(m0 + c0 + j) * p.N + gn) : 0u;
            }
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                // float(acc) / (cx * cw): true divide by the rounded product (oracle arithmetic)
                v[j] = __fdiv_rn((float)(int)r[j], __fmul_rn(cxs[c0 + j], cwn));
            }
            // outlier columns in list order, fp32 fma chain (oracle order)
            if (single_pass) {
                for (int t = 0; t < nj; ++t) {
                    const float wo = wos[t][row];
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = __fmaf_rn(xo[t][c0 + j], wo, v[j]);
                }
            } else {
                // many outliers: passes of kOJ columns staged through shared memory (all 128 threads take part)
                for (int t0 = 0; t0 < nj; t0 += kOJ) {
                    asm volatile("bar.sync 1, 128;" ::: "memory");      // previous pass fully read
                    stage_outliers(t0);
                    const int nt = min(kOJ, nj - t0);
                    for (int t = 0; t < nt; ++t) {
                        const float wo = wos[t][row];
#pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] = __fmaf_rn(xo[t][c0 + j], wo, v[j]);
                    }
                }
            }
            if (p.y_tma) {
                // [16 rows x 128 features] in the activation type -> one TMA store per chunk (rows past M and
                // features past N are clipped by the tensor map)
                uint16_t (*sb)[kOTileN] = ystage[(c0 >> 4) & 1];
                if (etid == 0 && c0 >= 32) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const ACT o = to_act<ACT>(v[j] + b);
                    sb[j][row] = *reinterpret_cast<const uint16_t*>(&o);
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (etid == 0 && c0 < m_valid) {
                    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                                 ::"l"(reinterpret_cast<uint64_t>(&tmap_y)), "r"(smem_u32(&sb[0][0])), "r"(n0), "r"(m0 + c0) : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            } else if (n_ok) {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (c0 + j < m_valid) y[(int64_t)(m0 + c0 + j) * p.N + gn] = to_act<ACT>(v[j] + b);
            }
        }
        if (p.y_tma && etid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}

// workspace: [flags K][colmax K uints][jcount + jlist (K+1 ints)][cx M floats][qx M*K bytes]
static size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

// split-K accumulator: only problems whose int32 result fits this region are split (small token counts)
constexpr size_t kOAccBytes = 4u << 20, kOCounterBytes = 16u << 10;

size_t int8_outlier_workspace_bytes(int64_t M, int64_t K) {
    return align256((size_t)K) + align256((size_t)K * 4) + kOCounterBytes + kOAccBytes + align256((size_t)(K + 1) * 4) +
           align256((size_t)M * 4) + align256((size_t)M * (size_t)K) + 512;
}

template <typename ACT>
static int outlier_launch(const ACT* x, const int8_t* qw, const float* cw, float threshold, const ACT* bias, ACT* y,
                          int64_t M, int64_t N, int64_t K, void* workspace, size_t ws_bytes, cudaStream_t st) {
    if (ws_bytes < int8_outlier_workspace_bytes(M, K)) return QUANTA_EWORKSPACE;
    uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    uint8_t* flag = ws;
    // [colmax | tile counters | acc] are contiguous: one memset clears what this call needs of them
    unsigned int* colmax = reinterpret_cast<unsigned int*>(ws + align256((size_t)K));
    unsigned int* counters = reinterpret_cast<unsigned int*>(reinterpret_cast<uint8_t*>(colmax) + align256((size_t)K * 4));
    int* acc = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(counters) + kOCounterBytes);
    int* jcount = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(acc) + kOAccBytes);
    int* jlist = jcount + 1;
    float* cx = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(jcount) + align256((size_t)(K + 1) * 4));
    int8_t* qx = reinterpret_cast<int8_t*>(reinterpret_cast<uint8_t*>(cx) + align256((size_t)M * 4));

    // tiling first: the split-K decision sizes the memset
    OutlierParams p;
    p.M = (int)M; p.N = (int)N; p.K = (int)K;
    int mb = (int)((M + 15) / 16 * 16);
    if (mb > 256) mb = 256;
    const int64_t n_tiles_n = (N + kOTileN - 1) / kOTileN;
    // one tile per CTA: pick the batch tile (256 / 128 / 64) that minimises waves x per-tile cost, the cost
    // of a tile being its batch rows plus a fixed part (weight tile, pipeline fill) worth ~64 rows
    if (mb > 64) {
        int best = mb;
        int64_t best_cost = -1;
        for (int cand = mb; cand >= 64 && cand % 16 == 0; cand /= 2) {
            const int64_t tiles = n_tiles_n * ((M + cand - 1) / cand);
            const int64_t cost = ((tiles + kNumSMs - 1) / kNumSMs) * (cand + 64);
            if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = cand; }
            if (cand % 32 != 0) break;
        }
        mb = best;
    }
    p.mb = mb;
    // split K while SMs would idle: small batches only (the int32 accumulator region is fixed-size)
    const int64_t tiles = n_tiles_n * ((M + mb - 1) / mb);
    const int nk_all = (int)((K + kOBlockK - 1) / kOBlockK);
    int splits = 1;
    // (measured: pays off for long K only — at K = 4096 the larger memset and the atomics cost more than the
    // shorter main loop saves: 20.3 -> 23.2 us at one token on 4096 x 4096, but 51.7 -> 42.8 us at K = 16384)
    if (nk_all >= 64 && (size_t)M * (size_t)N * 4 <= kOAccBytes && tiles * 4 <= (int64_t)kOCounterBytes) {
        while (splits < 16 && tiles * (splits * 2) <= kNumSMs && nk_all / (splits * 2) >= 4) splits *= 2;
    }
    p.splits = splits;
    if (splits > 1 || M > 64) {
        size_t clear = (size_t)K * 4;
        if (splits > 1) clear = align256((size_t)K * 4) + kOCounterBytes + (size_t)M * (size_t)N * 4;
        cudaError_t me = cudaMemsetAsync(colmax, 0, clear, st);
        if (me != cudaSuccess) return (int)me;
    }
    outlier_colmax_kernel<ACT><<<dim3((unsigned)((K + 255) / 256), (unsigned)((M + 63) / 64)), 256, 0, st>>>(x, (int)M, (int)K, colmax);
    outlier_columns_kernel<<<1, 1024, 0, st>>>(colmax, (int)K, threshold, flag, jlist, jcount);
    if (K % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0)
        outlier_rowquant_vec_kernel<ACT><<<(unsigned)M, 256, 0, st>>>(x, (int)K, flag, cx, qx);
    else
        outlier_rowquant_kernel<ACT><<<(unsigned)M, 256, 0, st>>>(x, (int)K, flag, cx, qx);

    p.a_bytes = kOTileN * kOBlockK;
    p.b_bytes = (uint32_t)mb * kOBlockK;
    int stages = (int)((150u * 1024u) / (p.a_bytes + p.b_bytes));      // the epilogue's tables take ~58 KB of static shared memory
    if (stages > kOMaxStages) stages = kOMaxStages;
    p.stages = stages;
    int cols = 32; while (cols < mb) cols <<= 1;
    p.tmem_cols = cols;

    CUtensorMap tmap_w, tmap_x;
    int rc = make_tensor_map_2d(&tmap_w, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, qw, (uint64_t)K, (uint64_t)N, (uint64_t)K, kOBlockK,
                                kOTileN, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = make_tensor_map_2d(&tmap_x, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, qx, (uint64_t)K, (uint64_t)M, (uint64_t)K, kOBlockK,
                            (uint32_t)mb, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    CUtensorMap tmap_y = tmap_w;                         // placeholder unless y can take TMA stores
    p.y_tma = ((reinterpret_cast<uintptr_t>(y) & 15) == 0 && (N & 7) == 0) ? 1 : 0;
    if (p.y_tma) {
        rc = make_tensor_map_2d(&tmap_y, sizeof(ACT) == 2 && std::is_same<ACT, __half>::value ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                                                                              : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
                                2, y, (uint64_t)N, (uint64_t)M, (uint64_t)N * 2, kOTileN, 16, CU_TENSOR_MAP_SWIZZLE_NONE);
        if (rc) return rc;
    }
    auto kern = int8_gemm_kernel<ACT>;
    const int smem = (int)(p.stages * (p.a_bytes + p.b_bytes) + kOEpiBytes + 1024);
    if (int e = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), smem)) return e;
    dim3 grid((unsigned)((N + kOTileN - 1) / kOTileN), (unsigned)((M + mb - 1) / mb), (unsigned)p.splits);
    kern<<<grid, kOThreads, smem, st>>>(tmap_w, tmap_x, tmap_y, x, qw, cw, cx, jlist, jcount, bias, y, acc, counters, p);
    return cuda_status(cudaGetLastError());
}

}  // namespace quanta

using namespace quanta;

extern "C" int quanta_int8_outlier_matmul(const void* x, int act_dtype, const int8_t* qw, const float* cw, float threshold,
                                          const void* bias, void* y, int64_t M, int64_t N, int64_t K, void* workspace,
                                          size_t workspace_bytes, void* stream) {
    if (!x || !qw || !cw || !y || !workspace || M <= 0 || N <= 0 || K <= 0) return QUANTA_EINVAL;
    if (K % 16 != 0) return QUANTA_EUNSUPPORTED;                                          // TMA row pitch
    if ((reinterpret_cast<uintptr_t>(qw) & 15) != 0) return QUANTA_EUNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (act_dtype == QUANTA_BF16)
        return outlier_launch<__nv_bfloat16>((const __nv_bfloat16*)x, qw, cw, threshold, (const __nv_bfloat16*)bias,
                                             (__nv_bfloat16*)y, M, N, K, workspace, workspace_bytes, st);
    if (act_dtype == QUANTA_F16)
        return outlier_launch<__half>((const __half*)x, qw, cw, threshold, (const __half*)bias, (__half*)y, M, N, K,
                                      workspace, workspace_bytes, st);
    return QUANTA_EINVAL;
}
