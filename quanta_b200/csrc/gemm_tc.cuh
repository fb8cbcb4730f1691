// Building blocks shared by the tcgen05 dequant-GEMM kernels: the forward y = x . dequant(W)^T
// (gemm.cu) and the input gradient dx = dy . dequant(W) (gemm_dgrad.cu).  Both dequantize with the
// same instructions, so the backward multiplies with bit-for-bit the weights the forward used.
#pragma once
#include "common.cuh"
#include "nf4_levels.cuh"

#include <cmath>

namespace quanta {

constexpr int kTileN = 128;          // output features per tile (UMMA M, TMEM lanes)
constexpr int kBlockK = 64;          // K per A slot / MMA group: one 128-byte swizzle atom of 16-bit activations
constexpr int kKbPerStage = 4;       // 64-K blocks per raw-code stage
constexpr int kStageK = kBlockK * kKbPerStage;
constexpr int kTmemCols = 512;
constexpr int kMaxRing = 12;
constexpr int kCounterBytes = 64 * 1024;     // per-tile arrival counters at the head of the workspace
constexpr int kMaxTiles = kCounterBytes / 4;

__device__ __forceinline__ uint4 lds128g(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t prmt_(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t r; asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel)); return r;
}
// (a & b) | c in one LOP3
__device__ __forceinline__ uint32_t and_or(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t r; asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r;
}
__device__ __forceinline__ void tma_load_2d_plain(uint32_t dst, const CUtensorMap* map, uint32_t bar, int32_t c0,
                                                  int32_t c1, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}

// ---- tcgen05 wrappers -----------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem descriptor]
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// completes `bar` (one arrival) when all previously issued MMAs of this thread have finished
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor: rows of 128 bytes, 8-row
// swizzle atoms 1024 bytes apart (SBO), LBO unused, descriptor version 1 (sm_100).
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

// ---- activation-type traits -------------------------------------------------
template <typename ACT> struct ActTraits;
template <> struct ActTraits<__nv_bfloat16> {
    static constexpr uint32_t kFmt = 1;                  // UMMA F16F32Format::BF16
    static constexpr uint32_t kMagic = 0x43004300u;      // bf16x2 (128 + n)
    static constexpr float kCentre = 136.0f;             // 128 + 8
    static constexpr CUtensorMapDataType kTma = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    using V2 = __nv_bfloat162;
    __device__ static __forceinline__ V2 dup(float v) { return __float2bfloat162_rn(v); }
    __device__ static __forceinline__ uint32_t pack(float a, float b) {
        V2 t = __floats2bfloat162_rn(a, b); return *reinterpret_cast<uint32_t*>(&t);
    }
    __device__ static __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
    __device__ static __forceinline__ __nv_bfloat16 from_float(float v) { return __float2bfloat16_rn(v); }
};
template <> struct ActTraits<__half> {
    static constexpr uint32_t kFmt = 0;                  // F16
    static constexpr uint32_t kMagic = 0x64006400u;      // fp16x2 (1024 + n)
    static constexpr float kCentre = 1032.0f;            // 1024 + 8
    static constexpr CUtensorMapDataType kTma = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    using V2 = __half2;
    __device__ static __forceinline__ V2 dup(float v) { return __float2half2_rn(v); }
    __device__ static __forceinline__ uint32_t pack(float a, float b) {
        V2 t = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&t);
    }
    __device__ static __forceinline__ float to_float(__half v) { return __half2float(v); }
    __device__ static __forceinline__ __half from_float(float v) { return __float2half_rn(v); }
};

// 4-bit: one 32-bit word = nibbles n0..n7 = 8 consecutive K values (pack_4bit_tensor layout).
// (magic | nibble) is the 16-bit float 128+n (bf16) / 1024+n (fp16), exactly; subtracting the
// centre leaves n-8 exactly, and one packed fma gives (n-8)*s + (z+8s) = n*s + z with the scale
// and the block midpoint z+8s rounded to the activation type (the midpoint is near zero for
// weight-like data, so its rounding error is far below the final 16-bit rounding of the weight).
template <typename ACT>
__device__ __forceinline__ void dequant_word4(uint32_t w, typename ActTraits<ACT>::V2 s2, typename ActTraits<ACT>::V2 z2,
                                              typename ActTraits<ACT>::V2 c2, uint32_t* out) {
    using V2 = typename ActTraits<ACT>::V2;
    constexpr uint32_t kM = ActTraits<ACT>::kMagic;
    uint32_t t[4];
    t[0] = and_or(w, 0x000F000Fu, kM);             // (n0, n4)
    t[1] = and_or(w >> 4, 0x000F000Fu, kM);        // (n1, n5)
    t[2] = and_or(w >> 8, 0x000F000Fu, kM);        // (n2, n6)
    t[3] = and_or(w >> 12, 0x000F000Fu, kM);       // (n3, n7)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        V2 v = *reinterpret_cast<V2*>(&t[i]);
        v = __hfma2(__hsub2(v, c2), s2, z2);
        t[i] = *reinterpret_cast<uint32_t*>(&v);
    }
    out[0] = prmt_(t[0], t[1], 0x5410u);           // (k0, k1)
    out[1] = prmt_(t[2], t[3], 0x5410u);           // (k2, k3)
    out[2] = prmt_(t[0], t[1], 0x7632u);           // (k4, k5)
    out[3] = prmt_(t[2], t[3], 0x7632u);           // (k6, k7)
}

// 8-bit: PRMT drops a code byte into bits 8..15 of 0x47000000, i.e. builds the fp32 value
// 32768 + q exactly; fma with zc = z - 32768*s gives q*s + z to within 2^-9 of a scale step,
// far inside the 16-bit rounding that follows (the reference rounds mul and add separately).
template <typename ACT>
__device__ __forceinline__ void dequant_word8(uint32_t w, float s, float zc, uint32_t* out) {
    float f[4];
#pragma unroll
    for (int e = 0; e < 4; ++e)
        f[e] = __fmaf_rn(__uint_as_float(prmt_(w, 0x47000000u, 0x7504u | (e << 4))), s, zc);
    out[0] = ActTraits<ACT>::pack(f[0], f[1]);
    out[1] = ActTraits<ACT>::pack(f[2], f[3]);
}

constexpr int kMaxOut = 8;
// NOUT = 1 for the plain GEMM (one map, compile-time loops), kMaxOut for the scatter entry
template <int NOUT>
struct GemmOutputs {
    CUtensorMap maps[NOUT];         // TMA-store maps of the output buffers ([M, col0 + N] windows, pitch ldy)
    void* y[NOUT];
};

struct GemmParams {
    int M, N, K;
    int mb;                 // UMMA N: batch rows per tile (multiple of 16, <= 256)
    int n_tiles, m_tiles;
    int total_kb;           // K / 64
    int S;                  // raw-code stages per tile: ceil(total_kb / 4)
    int G;                  // CTAs
    unsigned int U;         // work units: tiles * S  (U * G < 2^32, checked on the host)
    unsigned int uq, ur;    // U / G, U % G: CTA c owns units [c uq + min(c, ur), + uq + (c < ur))
    unsigned int s_magic;   // ceil(2^32 / S) (0: S == 1): u / S without a division — a 32-bit division is ~100
    unsigned int nt_magic;  // ceil(2^32 / n_tiles) (0: n_tiles == 1)   instructions on every role's critical path
    int nbuf;               // accumulator buffers in TMEM (1 or 2)
    int nacc;               // independent accumulators per buffer (power of 2): consecutive MMAs rotate over them
    int raw_stages, x_stages;
    int xkb;                // 64-K blocks per activation slot: 4, 2 or 1 (slot <= 32 KB)
    uint32_t raw_bytes, x_kb_bytes, x_slot_bytes, x_ring_off;
    int scale_stride;       // K / block
    int block_shift;        // log2(block / 64)
    int vec4;               // scale / zero-point rows can be read as float4 per stage
    int vec_store;          // 8-byte stores of 4 outputs are aligned in every output buffer
    int y_tma;              // whole tiles leave through a TMA store (needs N % 8 == 0 and an aligned y)
    int n_out;              // output buffers (1, or one per tensor-parallel peer: the tile is written to all of them)
    int ldy;                // row pitch of y in elements (N, or the full out_features of a column-parallel layer)
    int col0;               // first output column of this call inside y
    int nf4;                // 4-bit codes index the NF4 table, `scale` holds abs_max per block, zero-point unused
};

// Division-free index arithmetic (exactness of the multiplications is checked on the host, gemm_launch).
__device__ __forceinline__ unsigned int div_magic(unsigned int u, unsigned int magic) { return magic ? __umulhi(u, magic) : u; }
__device__ __forceinline__ unsigned int first_unit(unsigned int c, const GemmParams& p) { return c * p.uq + (c < p.ur ? c : p.ur); }
__device__ __forceinline__ int tile_of_unit(unsigned int u, const GemmParams& p) { return (int)div_magic(u, p.s_magic); }
// tile -> (n tile, m tile): tiles are numbered n-fastest
__device__ __forceinline__ void split_tile(int tile, const GemmParams& p, int& n_idx, int& m_idx) {
    m_idx = (int)div_magic((unsigned int)tile, p.nt_magic);
    n_idx = tile - m_idx * p.n_tiles;
}

// Contiguous range of work units of one CTA, walked tile by tile.
struct SegWalk {
    unsigned int u, u1, S, magic;
    __device__ __forceinline__ void init(const GemmParams& p, unsigned int cta) {
        u = first_unit(cta, p); u1 = first_unit(cta + 1u, p); S = (unsigned int)p.S; magic = p.s_magic;
    }
    // next segment: stages [s0, s1) of `tile`; false when the range is exhausted
    __device__ __forceinline__ bool next(int& tile, int& s0, int& s1) {
        if (u >= u1) return false;
        const unsigned int t = div_magic(u, magic);
        const unsigned int b = u - t * S, left = u1 - u;
        tile = (int)t; s0 = (int)b;
        s1 = (left < S - b) ? (int)(b + left) : (int)S;
        u += (unsigned int)(s1 - s0);
        return true;
    }
};

// CTA whose unit range contains unit `u`
__device__ __forceinline__ int cta_of_unit(unsigned int u, const GemmParams& p) {
    const unsigned int big = p.ur * (p.uq + 1u);
    return (int)(u < big ? u / (p.uq + 1u) : p.ur + (u - big) / p.uq);      // reducers only, once per tile
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n" : "=r"(pred));
    return pred != 0;
}

// Stream-K fix-up of one tile by `nthreads` threads (thread j): sum the fp32 partials of every
// contributing CTA in a fixed order (deterministic), add the bias, write y.  Thread -> 4 consecutive
// features, rows j/32, j/32 + nthreads/32, ...; kFixRows rows (float4 each) in flight per contributor.
constexpr int kFixRows = 6;
template <typename ACT, int NOUT>
__device__ __noinline__ void fixup_reduce(const GemmParams& p, const GemmOutputs<NOUT>& outs, const ACT* __restrict__ bias,
                                             const float* __restrict__ partial, int tile, int j, int nthreads) {
    using AT = ActTraits<ACT>;
    int n_tile, m_tile;
    split_tile(tile, p, n_tile, m_tile);
    const int m0 = m_tile * p.mb;
    const int m_valid = min(p.mb, p.M - m0);
    const int f4 = 4 * (j & 31), mq = j >> 5, mstep = nthreads >> 5;
    const int gn4 = n_tile * kTileN + f4;
    float b4[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) b4[e] = (bias != nullptr && gn4 + e < p.N) ? AT::to_float(bias[gn4 + e]) : 0.0f;
    const bool vec_ok = p.vec_store && gn4 + 3 < p.N;
    const unsigned int tu0 = (unsigned int)tile * (unsigned int)p.S;
    const int c_first = cta_of_unit(tu0, p), c_last = cta_of_unit(tu0 + (unsigned int)p.S - 1u, p);
    const size_t slot_elems = (size_t)(kTileN * p.mb);
    for (int mb0 = mq; mb0 < m_valid; mb0 += kFixRows * mstep) {
        float4 acc[kFixRows];
#pragma unroll
        for (int i = 0; i < kFixRows; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int c = c_first; c <= c_last; ++c) {
            const int wc = (tile == tile_of_unit(first_unit((unsigned int)c, p), p)) ? 0 : 1;
            const float* src = partial + ((size_t)c * 2 + wc) * slot_elems + f4;
            float4 v[kFixRows];
#pragma unroll
            for (int i = 0; i < kFixRows; ++i) {
                const int m = mb0 + mstep * i;
                v[i] = (m < m_valid) ? __ldcg(reinterpret_cast<const float4*>(src + m * kTileN))
                                     : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int i = 0; i < kFixRows; ++i) { acc[i].x += v[i].x; acc[i].y += v[i].y; acc[i].z += v[i].z; acc[i].w += v[i].w; }
        }
#pragma unroll
        for (int i = 0; i < kFixRows; ++i) {
            const int m = mb0 + mstep * i;
            if (m < m_valid) {
                const float o[4] = {acc[i].x + b4[0], acc[i].y + b4[1], acc[i].z + b4[2], acc[i].w + b4[3]};
                for (int ob = 0; ob < (NOUT == 1 ? 1 : p.n_out); ++ob) {
                    ACT* dst = static_cast<ACT*>(outs.y[ob]) + (int64_t)(m0 + m) * p.ldy + p.col0 + gn4;
                    if (vec_ok) {
                        uint2 pk;
                        pk.x = AT::pack(o[0], o[1]);
                        pk.y = AT::pack(o[2], o[3]);
                        *reinterpret_cast<uint2*>(dst) = pk;
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; ++e) if (gn4 + e < p.N) dst[e] = AT::from_float(o[e]);
                    }
                }
            }
        }
    }
}

// ---- host side --------------------------------------------------------------

// Number of CTAs: every SM with equal contiguous unit
// ranges (stream-K), or tiles x s units whose ranges coincide with tile boundaries (s = 1: no
// partials at all).  Costs in SM cycles, from the measurements in DESIGN.md: a stage (256 K) costs
// the MMA warp ~600 cycles of barrier traffic plus 16 MMAs of max(70, mb/2) cycles each, the
// dequant groups ~930 cycles, and one SM pulls its raw codes and its share of the activation
// tiles (re-read by every tile) out of L2 at ~29 B/cycle; a partial costs its fp32 store, ~4000
// cycles of release/acquire latency and the last arriver's (latency-bound) reads of every
// contributor's tile.
static int choose_units(int tiles, int S, int mb, int raw_bytes) {
    const int max_units = kNumSMs;
    const long long U = (long long)tiles * S;
    const double mma = 600.0 + 16.0 * (mb / 2.0 > 70.0 ? mb / 2.0 : 70.0);
    const double pull = (512.0 * mb + raw_bytes) / 29.0;
    const double stage = fmax(fmax(mma, 930.0), pull);
    const double tile_io = (double)kTileN * mb * 4.0 / 32.0;
    int best = 1;
    double best_cost = -1.0;
    auto consider = [&](int G) {
        if (G < 1 || G > max_units || (long long)G > U) return;
        double cost = (double)((U + G - 1) / G) * stage;
        if (G != tiles) {
            const double contributors = (double)G / tiles < 2.0 ? 2.0 : (double)G / tiles + 1.0;
            cost += 4000.0 + 2.0 * tile_io * (1.0 + contributors);
            // ranges that do not coincide with tile boundaries give most CTAs TWO partial tiles (two
            // accumulator drains and partial stores, uneven contributor counts): measured ~6 tile
            // transfers slower than the tile-aligned split on 4096 x 14336 at M = 64 / 128 / 256
            if (G % tiles != 0) cost += 6.0 * tile_io;
        }
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = G; }
    };
    consider(tiles <= max_units ? tiles : 0);
    for (int s = 2; tiles * s <= max_units && s <= S; ++s) consider(tiles * s);
    consider((int)(U < max_units ? U : max_units));
    return best;
}

size_t gemm_workspace_bytes(int64_t M, int64_t N);

}  // namespace quanta
