// W4A16 / W8A16 / NF4A16 dequantize-then-matmul for decode-sized batches (M <= 16; rows G1/G2 and N1 of SURVEY §8):
//     y[M,N] = x[M,K] . dequant(Wq)[N,K]^T + bias,   Wq blockwise-64 along K (convention A) or NF4 codes + abs_max.
//
// At these batch sizes the op is a pure weight stream (SURVEY App. D: 5.7 us of HBM time for a
// 4096 x 14336 W4 matrix), so the kernel is built around the stream and keeps everything else
// off its critical path:
//
//   * one persistent CTA per SM.  A producer thread keeps a ring of TMA stages full.  A stage is 256 BYTES of codes
//     per weight row — two SWIZZLE_128B boxes of [128 rows x 128 B] — plus the stage's [128 x kBlk] scale and
//     zero-point tiles (kBlk = 8 blocks of 64 K for 4-bit codes, 4 for 8-bit), all on one mbarrier: HBM serves
//     256-byte row pieces at its full rate, 128-byte ones at ~75 % of it (SmGeom).  The producer touches weights only,
//     so it never waits for the previous kernel (programmatic dependent launch; see pdl_wait in common.cuh for why
//     that is sound).  It requests `window` stages until the first one has landed (the TMA unit works on all of its
//     outstanding copies at once), then keeps the whole ring in flight.  The (row tile, stage) units are cut into
//     contiguous ranges, one per CTA (stream-K); how many CTAs is a cost model on the host (gemm_small_launch_nb);
//   * 16 consumer warps drain the ring (warp = 32 weight rows x kBpw 64-K blocks of every stage, so a B fragment
//     read from shared memory serves two row slabs).  Codes are never dequantized one by one: LOP3 drops a nibble
//     pair into the mantissas of the 16-bit constant 128.0 (bf16) / 1024.0 (fp16) — exact integers C + n — and the
//     warp-level tensor-core MMA (mma.sync m16n8k16, fp32 accumulate) forms raw = sum_k (C + n_k) x_k over one 64-K
//     block; scale and zero-point are applied once per block on the accumulators:
//         y += s * raw + (z - C s) * sum_k x_k
//     i.e. 7 integer instructions per 8 weights + 2 FMAs per accumulator, instead of 19 instructions per 8 weights
//     for an element-wise dequantization.  The MMA's K order is free as long as both operands agree, so x is staged
//     in the order the LOP3 pairs come out (k0,k4 | k1,k5 | k2,k6 | k3,k7) and no PRMT is needed.  8-bit codes go
//     through PRMT -> fp32 (32768 + q) -> q -> packed 16-bit, exact as well; NF4 codes through a byte -> level-pair
//     table in shared memory (one copy per lane), y += abs_max * raw;
//   * four staging warps read the stage's activations straight from global memory (L2), two to six units ahead in
//     registers, and write MMA fragment order plus the per-block sums of x into a ring of their own (full / empty
//     mbarriers), so the consumers' instruction stream is the weight path only and reads shared memory only;
//   * a CTA that covers only part of a row tile's K range stores an fp32 partial and bumps the tile's counter with
//     ONE fire-and-forget release; the CTA that owns the tile's last K steps is its reducer: once its own stream has
//     ended it acquires the counter, sums the partials in CTA order (deterministic), adds the bias and writes y — to
//     every output buffer of a tensor-parallel call (peer-mapped buffers over NVLink).  Nobody pays an atomic round
//     trip between two fences at the end of the kernel (measured 5-9 K cycles per CTA); when a range holds whole
//     tiles its partial segments are processed first, so the kernel ends on a plain store of y;
//   * no integer division anywhere in the kernel: unit ranges are c q + min(c, r), u / S a multiplication by a
//     host-computed reciprocal (a 32-bit division is ~100 instructions; they used to sit in every role's prologue
//     and cost 1.7 us per call).
//
// The products use the exact fp32 value q*s + z of the weight (the tcgen05 path in gemm.cu rounds it
// to the activation type first, like the reference's `.to(x.dtype)`); the difference is far inside
// the 1e-2 tolerance of rows G1/G2.
#include "common.cuh"
#include "nf4_levels.cuh"

#include <type_traits>

namespace quanta {

constexpr int kSmRows = 128;               // weight rows per tile
constexpr int kSmConsWarps = 16;           // warp w: rows 32 (w & 3) .. +32, block (w >> 2) of every step
constexpr int kSmConsThreads = 32 * kSmConsWarps;
// Activation staging warps: 4 — or 2 for a single batch row: 20 warps instead of 22 is one warp-allocation granule less,
// 96 instead of 80 registers per thread for the consumers, and two warps stage one row of x with time to spare
// (M = 1: 11.9 -> 11.8 / 11.4 -> 11.1 us W4, 16.2 -> 15.8 W8, 14.1 -> 13.6 NF4; at M = 8 two warps are too few: 14.1 us).
constexpr int sm_threads(int xw) { return kSmConsThreads + 64 + 32 * xw; }   // consumers + producer + publisher + staging warps
constexpr int kSmKGran = 256;              // K must be a multiple of this (16-byte scale rows; a partial last step is zero-filled)
constexpr int kSmMaxRing = 8;
constexpr int kSmMaxXRing = 4;             // activation slots (one stage each)
constexpr int kSmStartWindow = 2;          // stages requested before the first one has landed
constexpr int kSmMaxM = 16;                // batch rows served (NB = 2 column blocks of 8)
constexpr int kSmMaxOut = 8;
constexpr int kSmCounterBytes = 64 * 1024; // same workspace header as gemm.cu (zero before, zero after)

// One stage = 256 BYTES of codes per weight row (two SWIZZLE_128B boxes of [128 rows x 128 B]): HBM serves 256-byte
// row pieces at its full rate, 128-byte ones (the 4-bit kernel's first form: 256 K per stage) at ~75 % of it
// (measured: 4.8 vs 6.7 TB/s in the steady state of this kernel).
template <int BITS, bool NF4 = false> struct SmGeom {
    static constexpr int kStepK = 2048 / BITS;                       // K values per stage: 512 (4-bit) / 256 (8-bit)
    static constexpr int kBlk = kStepK / 64;                         // 64-K blocks per stage: 8 / 4
    static constexpr int kBpw = kBlk / 4;                            // blocks per consumer warp and stage: 2 / 1
    static constexpr uint32_t kCodeBytes = 32768u;
    static constexpr uint32_t kParamTile = (uint32_t)(kSmRows * kBlk * 4);   // one [128 rows x kBlk] fp32 tile
    static constexpr uint32_t kStageBytes = kCodeBytes + (NF4 ? 1u : 2u) * kParamTile;   // codes | scales (NF4: abs_max) | zero-points
};
constexpr uint32_t kSmLutBytes = 256u * 128u;   // NF4: byte -> (level[lo nibble], level[hi nibble]) in the activation type, one copy per lane

// Timeline of one launch (-DQUANTA_SMALL_TRACE build only): per CTA 40 clock64 stamps relative to kernel entry, + globaltimer at
// entry / exit in slots 38 / 39.  Read back with quanta_debug_small_trace().
#ifdef QUANTA_SMALL_TRACE
__device__ long long g_sm_trace[kNumSMs][40];
#define SM_TRACE(slot) do { if ((slot) < 38) g_sm_trace[blockIdx.x][(slot)] = clock64() - t_entry; } while (0)
#else
#define SM_TRACE(slot) do { } while (0)
#endif

struct SmallParams {
    int M, N, K;
    int S;                  // stages (SmGeom::kStepK K values) per row tile; the last one may be partial
    int n_tiles;
    int G;                  // CTAs
    unsigned int U;         // units = n_tiles * S
    unsigned int q, r;      // U / G, U % G: CTA c owns units [c q + min(c, r), + q + (c < r))
    unsigned int s_magic;   // ceil(2^32 / S): u / S == __umulhi(u, s_magic) for every u <= U (gemm_small_eligible); 0: S == 1
    int m_pad;              // 8 * NB
    int R;                  // weight ring stages
    int XR;                 // activation ring slots (<= kSmMaxXRing)
    int window;             // stages requested before the first one has landed (kSmStartWindow, at most R)
    int ldy, col0, n_out;
    int vec_y;              // 8-byte y stores are aligned in every output buffer
    uint32_t x_off;         // x ring
    uint32_t x_slot_bytes;  // NB * kBlk * (1024 fragment bytes + 32 block-sum bytes)
    uint32_t lut_off;       // NF4 pair table (kSmLutBytes), unused otherwise
    uint32_t red_off;       // [3][4 row groups][2 slabs][NB][4][32] floats: the K quarters of a tile meet here
    uint32_t bar_off;       // mbarriers + flags
    void* y[kSmMaxOut];
    // tensor-parallel completion inside the kernel (PeerSync, common.cuh); sync_world == 0: off
    unsigned int* sync_flags[kSmMaxOut];
    int sync_rank, sync_world;
    unsigned int* sync_epoch;   // this rank's call counter (local device memory)
};
constexpr int kSmDoneIdx = kSmCounterBytes / 4 - 1;          // the grid's exit counter for that (last word of the counter block)

template <typename ACT> struct SmTraits;
template <> struct SmTraits<__nv_bfloat16> {
    static constexpr uint32_t kMagic = 0x43004300u;   // bf16x2 (128 + n)
    static constexpr float kOffset = 128.0f;
    __device__ static __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
    __device__ static __forceinline__ __nv_bfloat16 from_float(float v) { return __float2bfloat16_rn(v); }
    __device__ static __forceinline__ uint32_t pack(float lo, float hi) {
        __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi); return *reinterpret_cast<uint32_t*>(&t);
    }
    __device__ static __forceinline__ void mma(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
        asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                     : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
    }
};
template <> struct SmTraits<__half> {
    static constexpr uint32_t kMagic = 0x64006400u;   // fp16x2 (1024 + n)
    static constexpr float kOffset = 1024.0f;
    __device__ static __forceinline__ float to_float(__half v) { return __half2float(v); }
    __device__ static __forceinline__ __half from_float(float v) { return __float2half_rn(v); }
    __device__ static __forceinline__ uint32_t pack(float lo, float hi) {
        __half2 t = __floats2half2_rn(lo, hi); return *reinterpret_cast<uint32_t*>(&t);
    }
    __device__ static __forceinline__ void mma(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
        asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                     : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
    }
};

__device__ __forceinline__ uint32_t sm_and_or(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t r; asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r;
}
__device__ __forceinline__ uint32_t sm_prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t r; asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel)); return r;
}
__device__ __forceinline__ uint2 sm_lds64(uint32_t addr) {
    uint2 v; asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr)); return v;
}
__device__ __forceinline__ uint4 sm_lds128(uint32_t addr) {
    uint4 v; asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sm_sts128(uint32_t addr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sm_sts32(uint32_t addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ float sm_lds32(uint32_t addr) {
    float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr)); return v;
}
__device__ __forceinline__ void sm_tma_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int32_t c0, int32_t c1, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void sm_bar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void sm_bar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "SMW_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra SMD_%=;\n\t"
        "bra SMW_%=;\n\t"
        "SMD_%=:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void sm_cons_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kSmConsThreads) : "memory"); }

// 4-bit: one 32-bit word = nibbles n0..n7 of 8 consecutive K values.  Four LOP3 (+ three shifts)
// give the exact 16-bit pairs (C+n0, C+n4), (C+n1, C+n5), (C+n2, C+n6), (C+n3, C+n7).
template <typename ACT>
__device__ __forceinline__ void sm_pairs4(uint32_t w, uint32_t* p) {
    constexpr uint32_t kM = SmTraits<ACT>::kMagic;
    p[0] = sm_and_or(w, 0x000F000Fu, kM);
    p[1] = sm_and_or(w >> 4, 0x000F000Fu, kM);
    p[2] = sm_and_or(w >> 8, 0x000F000Fu, kM);
    p[3] = sm_and_or(w >> 12, 0x000F000Fu, kM);
}
// 8-bit: one word = 4 codes; PRMT builds the fp32 value 32768 + q, one subtraction leaves q exactly,
// pairs (q0, q1), (q2, q3) in natural K order.
template <typename ACT>
__device__ __forceinline__ void sm_pairs8(uint32_t w, uint32_t* p) {
    float f[4];
#pragma unroll
    for (int e = 0; e < 4; ++e)
        f[e] = __fadd_rn(__uint_as_float(sm_prmt(w, 0x47000000u, 0x7504u | (e << 4))), -32768.0f);
    p[0] = SmTraits<ACT>::pack(f[0], f[1]);
    p[1] = SmTraits<ACT>::pack(f[2], f[3]);
}

// Row of the warp's 16-row slab that MMA row `gid` (0..7; +8 for the second half) stands for, chosen so
// that the shared-memory reads of the swizzled code tile are conflict-free: 4-bit reads 8 bytes per
// lane (a half-warp = MMA rows 0..3 must differ in bits 1-2 of the row), 8-bit 16 bytes per lane (a
// quarter-warp = MMA rows 2q, 2q+1 must differ in bit 2).
template <int BITS> __device__ __forceinline__ int sm_row_of(int gid) {
    return BITS == 4 ? (((gid & 3) << 1) | (gid >> 2)) : (((gid & 1) << 2) | (gid >> 1));
}

// The unit range of CTA c, and the CTA whose range contains unit u.  No division on the prologue's path: a 32-bit
// division is ~100 instructions and every CTA's first TMA request waits for it.
__device__ __forceinline__ unsigned int sm_first_unit(unsigned int c, const SmallParams& p) {
    return c * p.q + (c < p.r ? c : p.r);
}
__device__ __forceinline__ unsigned int sm_div_magic(unsigned int u, unsigned int magic) { return magic ? __umulhi(u, magic) : u; }
__device__ __forceinline__ unsigned int sm_div_S(unsigned int u, const SmallParams& p) { return sm_div_magic(u, p.s_magic); }
__device__ __forceinline__ int sm_cta_of_unit(unsigned int u, const SmallParams& p) {
    const unsigned int big = p.r * (p.q + 1u);
    return (int)(u < big ? u / (p.q + 1u) : p.r + (u - big) / p.q);
}

// The segments of a CTA's unit range [u0, u1) — a segment = this CTA's steps [s0, s1) of one row tile — in
// PROCESSING order.  A segment that covers only part of a tile's K range ends with a hand-over through global
// memory, a whole tile ends with a plain store of y.  So when the range holds whole tiles, the partial segments
// (the tail of the first tile, the head of the last one) are processed FIRST and handed over while the stream
// runs on, and the kernel ends on a whole tile.  With no whole tile in the range the natural order is kept.
struct SmWalk {
    unsigned int rb[3], re[3], u, S, magic;
    int nr, r;
    __device__ __forceinline__ void init(unsigned int u0, unsigned int u1, unsigned int S_, unsigned int magic_) {
        S = S_; magic = magic_; r = 0; nr = 0;
        const unsigned int t0 = sm_div_magic(u0, magic), tl = sm_div_magic(u1 - 1u, magic);
        const bool f_part = (u0 - t0 * S) != 0u && t0 != tl;            // tail of the first tile
        const bool l_part = (u1 - tl * S) != S && t0 != tl;             // head of the last tile
        const unsigned int wb = f_part ? (t0 + 1u) * S : u0, we = l_part ? tl * S : u1;
        if (t0 != tl && we > wb) {
            if (l_part) { rb[nr] = tl * S; re[nr] = u1; ++nr; }
            if (f_part) { rb[nr] = u0; re[nr] = (t0 + 1u) * S; ++nr; }
            rb[nr] = wb; re[nr] = we; ++nr;
        } else {
            rb[0] = u0; re[0] = u1; nr = 1;
        }
        u = rb[0];
    }
    // next segment: steps [s0, s1) of `tile`; `final`: nothing follows it
    __device__ __forceinline__ bool next(int& tile, int& s0, int& s1, bool& final) {
        if (r < nr && u >= re[r]) { ++r; if (r < nr) u = rb[r]; }
        if (r >= nr) return false;
        const unsigned int t = sm_div_magic(u, magic), b = u - t * S, left = re[r] - u;
        tile = (int)t; s0 = (int)b;
        s1 = (left < S - b) ? (int)(b + left) : (int)S;
        u += (unsigned int)(s1 - s0);
        final = (r == nr - 1) && u >= re[r];
        return true;
    }
};

// Stream-K hand-over of one tile.  The CTA that owns the tile's LAST K steps is its reducer; every other
// contributor stores its partial and bumps the tile's counter with ONE fire-and-forget release
// (red.release.gpu: the partial stores of the CTA — ordered before it by a CTA-level barrier — are visible to
// whoever acquires the incremented value).  The reducer's own share of the tile is the first thing it
// processes, so by the time its stream has ended the others have usually long arrived; it acquires the counter
// (bounded spin; contributors have lower CTA indices and were dispatched earlier), resets it for the next call
// and sums the partials.  A contributor never waits for anybody.
__device__ __forceinline__ void sm_contribute(unsigned int* counters, int tile) {
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counters + tile) : "memory");
}
__device__ __forceinline__ void sm_await_contributors(unsigned int* counters, int tile, int others) {
    unsigned int seen = 0, spins = 0;
    for (;;) {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counters + tile) : "memory");
        if (seen >= (unsigned int)others || ++spins > (1u << 22)) break;
    }
    counters[tile] = 0u;                                     // leave the workspace clean for the next call
}

// Sum the partials of every contributor of `tile` in CTA order (deterministic), add the bias, write y.
// Thread j of `nthreads` (a multiple of 32): 4 consecutive features, batch rows j / 32 + (nthreads / 32) k;
// 8 contributors' loads in flight per thread.
template <typename ACT>
__device__ __forceinline__ void sm_fixup(const SmallParams& p, const ACT* __restrict__ bias, const float* __restrict__ partial,
                                         int tile, int c_first, int c_last, int j, int nthreads) {
    using T = SmTraits<ACT>;
    const int n0 = tile * kSmRows;
    const int f4 = 4 * (j & 31), gn4 = n0 + f4;
    const size_t slot = (size_t)(kSmRows * p.m_pad);
    float b4[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) b4[e] = (bias != nullptr && gn4 + e < p.N) ? T::to_float(bias[gn4 + e]) : 0.0f;
    for (int m = j >> 5; m < p.M; m += nthreads >> 5) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int c0 = c_first; c0 <= c_last; c0 += 8) {
            float4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int c = c0 + u;
                v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (c <= c_last) {
                    const int wc = (tile == (int)sm_div_S(sm_first_unit((unsigned int)c, p), p)) ? 0 : 1;
                    v[u] = __ldcg(reinterpret_cast<const float4*>(partial + ((size_t)c * 2 + wc) * slot + m * kSmRows + f4));
                }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
        }
        const float o4[4] = {acc.x + b4[0], acc.y + b4[1], acc.z + b4[2], acc.w + b4[3]};
        for (int o = 0; o < p.n_out; ++o) {
            ACT* dst = static_cast<ACT*>(p.y[o]) + (int64_t)m * p.ldy + p.col0 + gn4;
            if (p.vec_y && gn4 + 3 < p.N) {
                uint2 pk;
                pk.x = T::pack(o4[0], o4[1]);
                pk.y = T::pack(o4[2], o4[3]);
                *reinterpret_cast<uint2*>(dst) = pk;
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) if (gn4 + e < p.N) dst[e] = T::from_float(o4[e]);
            }
        }
    }
}

template <typename ACT, int BITS, int NB, bool NF4, int XW>
__global__ void __launch_bounds__(sm_threads(XW), 1)
gemm_small_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_s,
                  const __grid_constant__ CUtensorMap tmap_z, const ACT* __restrict__ x, const ACT* __restrict__ bias,
                  unsigned int* __restrict__ counters, float* __restrict__ partial, const __grid_constant__ SmallParams p) {
    using T = SmTraits<ACT>;
    using G = SmGeom<BITS, NF4>;
    static_assert(!NF4 || BITS == 4, "NF4 codes are 4-bit");
    constexpr int kSmXWarps = XW, kSmThreads = sm_threads(XW);
    extern __shared__ __align__(1024) uint8_t sm_raw[];

    const uint32_t smem = smem_u32(sm_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const uint32_t bars = smem + p.bar_off;                  // full[R] | empty[R] | xfull[XR] | xempty[XR]
    auto full_bar = [&](int s) { return bars + (uint32_t)s * 8u; };
    auto empty_bar = [&](int s) { return bars + (uint32_t)(kSmMaxRing + s) * 8u; };
    auto xfull_bar = [&](int s) { return bars + (uint32_t)(2 * kSmMaxRing + s) * 8u; };
    auto xempty_bar = [&](int s) { return bars + (uint32_t)(2 * kSmMaxRing + kSmMaxXRing + s) * 8u; };

#ifdef QUANTA_SMALL_TRACE
    const long long t_entry = clock64();
    if (tid == 0) { unsigned long long g; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g)); g_sm_trace[blockIdx.x][38] = (long long)g; }
#endif
    const unsigned int cta = blockIdx.x;
    const unsigned int u0 = sm_first_unit(cta, p), u1 = sm_first_unit(cta + 1u, p);
    const int S = p.S;
    const int tile0 = (int)sm_div_S(u0, p);              // the first tile of the range owns partial slot 0
    SmWalk walk;
    walk.init(u0, u1, (unsigned int)S, p.s_magic);
    int tile, s0, s1;
    bool final_seg;

    // The producer initialises the weight ring itself, checks in at the CTA barrier WITHOUT waiting (bar.arrive)
    // and starts streaming at once; everybody else sees all barriers after bar.sync.
    if (tid == 32 * kSmConsWarps) {
        SM_TRACE(32);
        prefetch_tensormap(&tmap_w); prefetch_tensormap(&tmap_s); prefetch_tensormap(&tmap_z);
        for (int s = 0; s < p.R; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(full_bar(s)), "r"(1));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(empty_bar(s)), "r"(kSmConsWarps));
        }
        fence_barrier_init();
        SM_TRACE(33);
    }
    if (tid == 0) {
        for (int s = 0; s < kSmMaxXRing; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(xfull_bar(s)), "r"(kSmXWarps));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(xempty_bar(s)), "r"(kSmConsWarps));
        }
        fence_barrier_init();
    }
    if (warp == kSmConsWarps) {
        __syncwarp();
        asm volatile("barrier.arrive 0, %0;" ::"n"(kSmThreads) : "memory");
    } else {
        asm volatile("barrier.sync 0, %0;" ::"n"(kSmThreads) : "memory");
    }

    if (warp == kSmConsWarps) {
        // ===== producer: keeps the ring full across tile boundaries =====
        // Programmatic dependent launch: this grid may start while the previous kernel on the stream is still in its
        // tail.  The producer touches only the weight operands, which do not depend on that kernel (common.cuh,
        // pdl_wait), so it never waits for it; the activations and every global write of this grid are ordered
        // behind griddepcontrol.wait in the other warps.
        if (lane == 0) {
            SM_TRACE(34);
            const uint64_t pol = policy_evict_first();       // weights are streamed once
            int slot = 0, i = 0;
            uint32_t ph = 0;
            while (walk.next(tile, s0, s1, final_seg)) {
                for (int step = s0; step < s1; ++step, ++i) {
                    if (i == 0) SM_TRACE(1);
                    if (i == p.window) {
                        // start-up window: the TMA unit works on all of its outstanding copies at once, so the first
                        // stage lands sooner when only a few are requested; the whole ring opens once it is there
                        SM_TRACE(2);
                        sm_bar_wait(full_bar(0), 0u);
                        SM_TRACE(3);
                    }
                    if (i >= p.R) sm_bar_wait(empty_bar(slot), ph ^ 1u);
                    const uint32_t bar = full_bar(slot);
                    const uint32_t dst = smem + (uint32_t)slot * G::kStageBytes;
                    const int kb = step * G::kStepK, n0 = tile * kSmRows;
                    const int cb = kb * BITS / 8;            // byte column of the stage in a code row
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(G::kStageBytes) : "memory");
                    sm_tma_2d(dst, &tmap_w, bar, cb, n0, pol);
                    sm_tma_2d(dst + 16384u, &tmap_w, bar, cb + 128, n0, pol);
                    sm_tma_2d(dst + G::kCodeBytes, &tmap_s, bar, kb / 64, n0, pol);
                    if (!NF4) sm_tma_2d(dst + G::kCodeBytes + G::kParamTile, &tmap_z, bar, kb / 64, n0, pol);
                    if (++slot == p.R) { slot = 0; ph ^= 1u; }
                }
            }
            SM_TRACE(4);
        }
        return;
    }
    // Let the next kernel on the stream start its own prologue as soon as this grid's CTAs make room (its weights do
    // not depend on us).  Every warp orders its GLOBAL accesses behind the previous kernel (griddepcontrol.wait): the
    // staging warps before they read x, the publisher before its first release, the consumers — which read shared
    // memory only — before the first store of a segment's result.  Their set-up runs ahead of the wait.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (warp == kSmConsWarps + 1) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        // ===== publisher: releases the partial of every contributor segment that is not the CTA's last one while
        //       the stream runs on (a segment that reaches the tile's last step makes this CTA the reducer: no release) =====
        while (walk.next(tile, s0, s1, final_seg)) {
            if (final_seg || s1 == S) continue;
            asm volatile("bar.sync 2, 160;" ::: "memory");   // the 4 output warps have stored the partial
            if (lane == 0) sm_contribute(counters, tile);
        }
        return;
    }

    if (warp >= kSmConsWarps + 2) {
        // ===== activation staging warps =====
        // They read the stage's activations x[0..m_pad) x [kStepK] straight from global memory (L2: every CTA reads the
        // same few hundred KB), one stage ahead in registers, and write them in MMA fragment order plus the per-block
        // sums of x into a ring of their own.  Chunk c (c = 32 xw + lane + 128 it) = 8 consecutive K values: batch row
        // m = c / kRowChunks, cc = c % kRowChunks -> block cc / 8, K offset 8 (cc & 7) within the block -> slot chunk
        // (((nb kBlk + blk) 2 + j) 32 + gid 4 + tig) with nb = m / 8, gid = m & 7, tig = (cc & 7) / 2, j = cc & 1: a
        // consumer warp's B-fragment read of one (nb, blk, j) is 512 contiguous bytes.
        constexpr int kRowChunks = G::kStepK / 8;            // 16-byte chunks per batch row and stage: 64 / 32
        constexpr int kChunks = 8 * NB * kRowChunks;
        constexpr int kPer = kChunks / (32 * kSmXWarps);     // chunks per thread and stage: 4 NB / 2 NB
        constexpr int kMStep = 32 * kSmXWarps / kRowChunks;  // batch rows between a thread's chunks: 2 / 4
        const int xw = warp - (kSmConsWarps + 2);
        // chunk `it` of this thread: batch row m_first + kMStep it, always the same cc
        const int c_first = 32 * xw + lane;
        const int m_first = c_first / kRowChunks, cc = c_first % kRowChunks, blk = cc >> 3, c8 = cc & 7;
        const uint32_t xdst0 = (uint32_t)(((blk * 2 + (c8 & 1)) * 32 + m_first * 4 + (c8 >> 1)) * 16);
        const uint32_t xsum0 = (uint32_t)(NB * G::kBlk * 1024 + (blk * 8 + m_first) * 4);
        const ACT* const xrow0 = x + (size_t)m_first * (size_t)p.K + cc * 8;
        const size_t row_step = (size_t)kMStep * (size_t)p.K;
        // Rows past M are zero in every slot, for ever: written once, here (ordered before the consumers' reads by the
        // first xfull arrive of this thread).
        for (uint32_t o = (uint32_t)(32 * xw + lane) * 16u; o < (uint32_t)p.XR * p.x_slot_bytes; o += 32u * kSmXWarps * 16u)
            sm_sts128(smem + p.x_off + o, make_uint4(0u, 0u, 0u, 0u));
        asm volatile("bar.sync 3, %0;" ::"n"(32 * kSmXWarps) : "memory");   // nobody's zeros land on a sibling's first unit
        const int n_units = (int)(u1 - u0);
        // RPT chunks per thread and unit are live (1 when M <= kMStep: then the thread's other chunks are padding rows),
        // DEPTH units are in flight in registers: an L2 round trip under the weight stream's load is 2-3 K cycles, and
        // right after the dependency wait — when up to R stages of weights are already waiting in shared memory — these
        // warps, not the stream, pace the consumers.
        auto stage_all = [&](auto rpt_tag, auto depth_tag) {
            constexpr int RPT = decltype(rpt_tag)::value, DEPTH = decltype(depth_tag)::value;
            uint4 buf[DEPTH][RPT];
            SmWalk ahead = walk;
            int a_tile, a_s0 = 0, a_s1 = 0, a_step = 0;
            bool a_fin, a_ok = ahead.next(a_tile, a_s0, a_s1, a_fin);
            a_step = a_s0;
            auto fetch_next = [&](uint4* dst) {
                if (!a_ok) return;
                const int k = a_step * G::kStepK;
                const bool k_ok = k + cc * 8 < p.K;          // false only in the K tail of a partial last stage
#pragma unroll
                for (int it = 0; it < RPT; ++it) {
                    dst[it] = make_uint4(0u, 0u, 0u, 0u);    // rows past M and that tail read as zero
                    if (k_ok && m_first + kMStep * it < p.M) dst[it] = __ldcg(reinterpret_cast<const uint4*>(xrow0 + it * row_step + k));
                }
                if (++a_step >= a_s1) { a_ok = ahead.next(a_tile, a_s0, a_s1, a_fin); a_step = a_s0; }
            };
            asm volatile("griddepcontrol.wait;" ::: "memory");   // x is the previous kernel's output
            if (xw == 0 && lane == 0) SM_TRACE(24);
#pragma unroll
            for (int d = 0; d < DEPTH; ++d) fetch_next(buf[d]);
            int xs = 0, i = 0;
            uint32_t ph = 0;
            while (i < n_units) {
#pragma unroll
                for (int d = 0; d < DEPTH; ++d) {
                    if (i >= n_units) break;
                    if (i >= p.XR) sm_bar_wait(xempty_bar(xs), ph ^ 1u);
                    const uint32_t slot = smem + p.x_off + (uint32_t)xs * p.x_slot_bytes;
#pragma unroll
                    for (int it = 0; it < RPT; ++it) {
                        const int mo = kMStep * it;          // compile-time: nb = mo / 8, row within the block of 8: (mo & 7) + m_first
                        uint4 v = buf[d][it];
                        const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
                        float sum = 0.0f;
                        if (SmTraits<ACT>::kOffset == 128.0f) {
                            // bf16 -> fp32 is a shift / mask
#pragma unroll
                            for (int q = 0; q < 4; ++q) sum += __uint_as_float(w4[q] << 16) + __uint_as_float(w4[q] & 0xFFFF0000u);
                        } else {
                            const ACT* e = reinterpret_cast<const ACT*>(&v);
#pragma unroll
                            for (int q = 0; q < 8; ++q) sum += T::to_float(e[q]);
                        }
                        sum += __shfl_xor_sync(0xffffffffu, sum, 1);
                        sum += __shfl_xor_sync(0xffffffffu, sum, 2);
                        sum += __shfl_xor_sync(0xffffffffu, sum, 4);
                        if (BITS == 4 && !NF4) {
                            uint4 o;
                            o.x = sm_prmt(v.x, v.z, 0x5410u);    // (x0, x4)
                            o.y = sm_prmt(v.x, v.z, 0x7632u);    // (x1, x5)
                            o.z = sm_prmt(v.y, v.w, 0x5410u);    // (x2, x6)
                            o.w = sm_prmt(v.y, v.w, 0x7632u);    // (x3, x7)
                            v = o;
                        }
                        sm_sts128(slot + xdst0 + (uint32_t)((mo >> 3) * G::kBlk * 1024 + (mo & 7) * 64), v);
                        if ((lane & 7) == 0) sm_sts32(slot + xsum0 + (uint32_t)((mo >> 3) * G::kBlk * 32 + (mo & 7) * 4), sum);
                    }
                    fetch_next(buf[d]);                      // unit i + DEPTH
                    __syncwarp();
                    if (lane == 0) sm_bar_arrive(xfull_bar(xs));
#ifdef QUANTA_SMALL_TRACE
                    if (xw == 0 && lane == 0 && i < 2) SM_TRACE(25 + i);
#endif
                    if (++xs == p.XR) { xs = 0; ph ^= 1u; }
                    ++i;
                }
            }
        };
        if (p.M <= kMStep) stage_all(std::integral_constant<int, 1>{}, std::integral_constant<int, 6>{});
        else stage_all(std::integral_constant<int, kPer>{}, std::integral_constant<int, (NB == 1 ? 2 : 1)>{});
        return;
    }

    // ===== consumers =====
    const int gid = lane >> 2, tig = lane & 3;
    const int rg = warp & 3, kq = warp >> 2;                 // rows 32 rg .. +32, blocks kBpw kq .. + kBpw of every stage
    // rows[sl][h]: slab sl (16 rows), MMA row gid + 8 h
    int rows[2][2];
#pragma unroll
    for (int sl = 0; sl < 2; ++sl) { rows[sl][0] = (2 * rg + sl) * 16 + sm_row_of<BITS>(gid); rows[sl][1] = rows[sl][0] + 8; }

    // Absolute shared-memory addresses of this thread's words in slot 0 (rows + 8 / + 16 keep the swizzle phase, so
    // every other address of a stage is one of these plus an immediate).  Made opaque so that they live in registers:
    // ptxas otherwise rematerialises the lane / warp arithmetic inside the stage loop.
    const int r00 = rows[0][0];
    uint32_t w_base[G::kBpw];
#pragma unroll
    for (int bb = 0; bb < G::kBpw; ++bb) {
        const int b = kq * G::kBpw + bb;                     // block of the stage
        const uint32_t off = BITS == 4
            ? (uint32_t)(b >> 2) * 16384u + (uint32_t)r00 * 128u + ((((uint32_t)(2 * (b & 3) + (tig >> 1))) ^ (uint32_t)(r00 & 7)) << 4) + (uint32_t)(tig & 1) * 8u
            : (uint32_t)(b >> 1) * 16384u + (uint32_t)r00 * 128u + ((((uint32_t)(4 * (b & 1) + tig)) ^ (uint32_t)(r00 & 7)) << 4);
        w_base[bb] = smem + off;
        asm volatile("" : "+r"(w_base[bb]));
    }
    constexpr uint32_t kRowPitch = (uint32_t)(G::kBlk * 4);  // bytes per row of a scale / zero-point tile
    uint32_t s_base = smem + G::kCodeBytes + (uint32_t)r00 * kRowPitch + (uint32_t)(kq * G::kBpw) * 4u;
    uint32_t xb_base = smem + p.x_off + (uint32_t)((kq * G::kBpw) * 1024 + lane * 16);
    uint32_t xs_base0 = smem + p.x_off + (uint32_t)(NB * G::kBlk * 1024 + ((kq * G::kBpw) * 8 + 2 * tig) * 4);
    asm volatile("" : "+r"(s_base), "+r"(xb_base), "+r"(xs_base0));
    const uint32_t x_slot_bytes = p.x_slot_bytes;
    const int ring = p.R, xring = p.XR;
    // NF4: the 16 levels are not an affine function of the code, so the exact-integer trick does not apply; a code BYTE
    // is looked up instead: table[b] = (level[b & 15], level[b >> 4]) as a 16-bit pair — the two K-adjacent weights of
    // the byte, in natural K order — replicated once per lane (entry b of lane l at b * 128 + 4 l: every lane of a
    // lookup hits its own bank).  2 ALU instructions + 1 LDS per byte instead of 7 ALU per word.
    uint32_t lut_lane = smem + p.lut_off + (uint32_t)lane * 4u;
    if (NF4) {
        for (int e = tid; e < 256 * 32; e += kSmConsThreads) {
            const int b = e >> 5;
            const uint32_t pr = T::pack(kNf4Levels[b & 15], kNf4Levels[b >> 4]);
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(smem + p.lut_off + (uint32_t)e * 4u), "r"(pr) : "memory");
        }
        sm_cons_sync();
        asm volatile("" : "+r"(lut_lane));
    }

    float tot[2][NB][4];
#pragma unroll
    for (int sl = 0; sl < 2; ++sl)
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) { tot[sl][nb][0] = tot[sl][nb][1] = tot[sl][nb][2] = tot[sl][nb][3] = 0.0f; }
    int wslot = 0, xs_cur = 0, red_tile = -1;
    uint32_t wph = 0, xph = 0;

#ifdef QUANTA_SMALL_TRACE
    int tr_unit = 0;
#endif
    if (tid == 0) SM_TRACE(5);
    while (walk.next(tile, s0, s1, final_seg)) {
        for (int step = s0; step < s1; ++step) {
            sm_bar_wait(full_bar(wslot), wph);
#ifdef QUANTA_SMALL_TRACE
            if (tid == 0 && tr_unit == 0) SM_TRACE(27);
#endif
            sm_bar_wait(xfull_bar(xs_cur), xph);
#ifdef QUANTA_SMALL_TRACE
            if (tid == 0 && tr_unit == 0) SM_TRACE(28);
#endif

            const uint32_t st_off = (uint32_t)wslot * G::kStageBytes, x_off = (uint32_t)xs_cur * x_slot_bytes;
            // scales / zero-points of the warp's blocks: rows (slab, half), kBpw adjacent blocks each
            // (M <= 8: both blocks in one 8-byte read up front; M > 8: per block, late — registers)
            constexpr bool kParamsUpFront = NB == 1;
            float sc[2][2][G::kBpw], zc[2][2][G::kBpw];
#pragma unroll
            for (int sl = 0; sl < 2; ++sl)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (!kParamsUpFront) break;
                    const uint32_t sa = s_base + st_off + (uint32_t)(sl * 16 + h * 8) * kRowPitch;
                    if (G::kBpw == 2) {
                        const uint2 a = sm_lds64(sa);
                        sc[sl][h][0] = __uint_as_float(a.x); sc[sl][h][G::kBpw - 1] = __uint_as_float(a.y);
                        if (!NF4) {
                            const uint2 z = sm_lds64(sa + G::kParamTile);
                            zc[sl][h][0] = __uint_as_float(z.x); zc[sl][h][G::kBpw - 1] = __uint_as_float(z.y);
                        }
                    } else {
                        sc[sl][h][0] = sm_lds32(sa);
                        if (!NF4) zc[sl][h][0] = sm_lds32(sa + G::kParamTile);
                    }
                }
            const float off = BITS == 4 ? T::kOffset : 0.0f;
#pragma unroll
            for (int bb = 0; bb < G::kBpw; ++bb) {
                // ---- every shared-memory read of the block goes out first (ordered asm statements; the
                //      arithmetic below is free for the compiler to interleave) ----
                const uint32_t w_cur = w_base[bb] + st_off;
                uint32_t wraw[2][2][BITS == 4 ? 2 : 4];  // [slab][row half][words]
#pragma unroll
                for (int sl = 0; sl < 2; ++sl)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const uint32_t wa = w_cur + (uint32_t)(sl * 2048 + h * 1024);
                        if (BITS == 4) {
                            const uint2 w = sm_lds64(wa);
                            wraw[sl][h][0] = w.x; wraw[sl][h][1] = w.y;
                        } else {
                            const uint4 w = sm_lds128(wa);
                            wraw[sl][h][0] = w.x; wraw[sl][h][1] = w.y; wraw[sl][h][BITS == 4 ? 0 : 2] = w.z; wraw[sl][h][BITS == 4 ? 1 : 3] = w.w;
                        }
                    }
                uint4 xb[NB];                            // the B fragments of two k steps; re-read for k = 2
                uint2 xs2[NB];
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) {
                    xb[nb] = sm_lds128(xb_base + x_off + (uint32_t)((nb * G::kBlk + bb) * 1024));
                    if (!NF4) xs2[nb] = sm_lds64(xs_base0 + x_off + (uint32_t)((nb * G::kBlk + bb) * 32));
                }
                // ---- 4 MMAs (K = 16 each) per slab and batch block: k outermost, so that consecutive MMAs
                //      are independent (2 slabs x NB accumulators) ----
                float c[2][NB][4];
#pragma unroll
                for (int sl = 0; sl < 2; ++sl)
#pragma unroll
                    for (int nb = 0; nb < NB; ++nb) { c[sl][nb][0] = c[sl][nb][1] = c[sl][nb][2] = c[sl][nb][3] = 0.0f; }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (k == 2) {
#pragma unroll
                        for (int nb = 0; nb < NB; ++nb) xb[nb] = sm_lds128(xb_base + x_off + (uint32_t)((nb * G::kBlk + bb) * 1024 + 512));
                    }
                    uint32_t a[2][4];                    // {row lo, row+8 lo, row hi, row+8 hi}
#pragma unroll
                    for (int sl = 0; sl < 2; ++sl) {
                        if (NF4) {
                            // word k / 2, bytes 2 (k & 1) and 2 (k & 1) + 1: K-adjacent pairs in natural order
                            const uint32_t r0 = wraw[sl][0][k >> 1], r1 = wraw[sl][1][k >> 1];
                            const uint32_t i00 = (k & 1) ? ((r0 >> 9) & 0x7F80u) : ((r0 << 7) & 0x7F80u);
                            const uint32_t i01 = (k & 1) ? ((r0 >> 17) & 0x7F80u) : ((r0 >> 1) & 0x7F80u);
                            const uint32_t i10 = (k & 1) ? ((r1 >> 9) & 0x7F80u) : ((r1 << 7) & 0x7F80u);
                            const uint32_t i11 = (k & 1) ? ((r1 >> 17) & 0x7F80u) : ((r1 >> 1) & 0x7F80u);
                            a[sl][0] = __float_as_uint(sm_lds32(lut_lane + i00));
                            a[sl][1] = __float_as_uint(sm_lds32(lut_lane + i10));
                            a[sl][2] = __float_as_uint(sm_lds32(lut_lane + i01));
                            a[sl][3] = __float_as_uint(sm_lds32(lut_lane + i11));
                        } else if (BITS == 4) {
                            // word k / 2: pairs (n0,n4) (n1,n5) for even k, (n2,n6) (n3,n7) for odd k.  (The shifts stay
                            // on the ALU pipe: as IMAD.HI they measured 25 % slower, tools/micro/unit_mix.cu.)
                            const uint32_t w0 = wraw[sl][0][k >> 1] >> (8 * (k & 1)), w1 = wraw[sl][1][k >> 1] >> (8 * (k & 1));
                            a[sl][0] = sm_and_or(w0, 0x000F000Fu, T::kMagic);
                            a[sl][1] = sm_and_or(w1, 0x000F000Fu, T::kMagic);
                            a[sl][2] = sm_and_or(w0 >> 4, 0x000F000Fu, T::kMagic);
                            a[sl][3] = sm_and_or(w1 >> 4, 0x000F000Fu, T::kMagic);
                        } else {
                            uint32_t p0[2], p1[2];
                            sm_pairs8<ACT>(wraw[sl][0][k], p0); sm_pairs8<ACT>(wraw[sl][1][k], p1);
                            a[sl][0] = p0[0]; a[sl][1] = p1[0]; a[sl][2] = p0[1]; a[sl][3] = p1[1];
                        }
                    }
#pragma unroll
                    for (int nb = 0; nb < NB; ++nb) {
                        const uint4 xv4 = xb[nb];
                        const uint32_t b0 = (k & 1) ? xv4.z : xv4.x, b1 = (k & 1) ? xv4.w : xv4.y;
#pragma unroll
                        for (int sl = 0; sl < 2; ++sl) T::mma(c[sl][nb], a[sl], b0, b1);
                    }
                }
#pragma unroll
                for (int sl = 0; sl < 2; ++sl) {
                    if (!kParamsUpFront) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            const uint32_t sa = s_base + st_off + (uint32_t)(sl * 16 + h * 8) * kRowPitch + (uint32_t)(bb * 4);
                            sc[sl][h][bb] = sm_lds32(sa);
                            if (!NF4) zc[sl][h][bb] = sm_lds32(sa + G::kParamTile);
                        }
                    }
                    if (NF4) {
                        // y += abs_max * raw: the table holds the levels themselves, no offset term
#pragma unroll
                        for (int nb = 0; nb < NB; ++nb) {
                            tot[sl][nb][0] = __fmaf_rn(sc[sl][0][bb], c[sl][nb][0], tot[sl][nb][0]);
                            tot[sl][nb][1] = __fmaf_rn(sc[sl][0][bb], c[sl][nb][1], tot[sl][nb][1]);
                            tot[sl][nb][2] = __fmaf_rn(sc[sl][1][bb], c[sl][nb][2], tot[sl][nb][2]);
                            tot[sl][nb][3] = __fmaf_rn(sc[sl][1][bb], c[sl][nb][3], tot[sl][nb][3]);
                        }
                        continue;
                    }
                    const float s_0 = sc[sl][0][bb], s_1 = sc[sl][1][bb];
                    const float z0 = __fmaf_rn(-off, s_0, zc[sl][0][bb]), z1 = __fmaf_rn(-off, s_1, zc[sl][1][bb]);
#pragma unroll
                    for (int nb = 0; nb < NB; ++nb) {
                        const float xs_a = __uint_as_float(xs2[nb].x), xs_b = __uint_as_float(xs2[nb].y);
                        tot[sl][nb][0] = __fmaf_rn(s_0, c[sl][nb][0], __fmaf_rn(z0, xs_a, tot[sl][nb][0]));
                        tot[sl][nb][1] = __fmaf_rn(s_0, c[sl][nb][1], __fmaf_rn(z0, xs_b, tot[sl][nb][1]));
                        tot[sl][nb][2] = __fmaf_rn(s_1, c[sl][nb][2], __fmaf_rn(z1, xs_a, tot[sl][nb][2]));
                        tot[sl][nb][3] = __fmaf_rn(s_1, c[sl][nb][3], __fmaf_rn(z1, xs_b, tot[sl][nb][3]));
                    }
                }
            }
            // every lane's reads of the stage have been issued (and, in program order, consumed) above
            __syncwarp();
            if (lane == 0) { sm_bar_arrive(empty_bar(wslot)); sm_bar_arrive(xempty_bar(xs_cur)); }
            if (++wslot == ring) { wslot = 0; wph ^= 1u; }
            if (++xs_cur == xring) { xs_cur = 0; xph ^= 1u; }
#ifdef QUANTA_SMALL_TRACE
            if (tid == 0 && tr_unit < 16) { SM_TRACE(8 + tr_unit); ++tr_unit; }
#endif
        }
        if (tid == 0) SM_TRACE(6);
        asm volatile("griddepcontrol.wait;" ::: "memory");   // the first global accesses of the consumers follow
        // ===== end of this CTA's segment [s0, s1) of `tile`: the 4 K quarters meet in shared memory =====
        const bool whole = s0 == 0 && s1 == S;
        const uint32_t red = smem + p.red_off + (uint32_t)(rg * (2 * NB * 4) * 128 + lane * 4);
        const uint32_t red_group = (uint32_t)(4 * 2 * NB * 4 * 128);
        if (kq > 0) {
#pragma unroll
            for (int sl = 0; sl < 2; ++sl)
#pragma unroll
                for (int nb = 0; nb < NB; ++nb)
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        sm_sts32(red + (uint32_t)(kq - 1) * red_group + (uint32_t)(((sl * NB + nb) * 4 + q) * 128), tot[sl][nb][q]);
        }
        sm_cons_sync();
        if (tid == 0) SM_TRACE(29);
        const int n0 = tile * kSmRows;
        if (kq == 0) {
            // tot[sl][nb][q]: feature n0 + rows[sl][q >> 1], batch row 8 nb + 2 tig + (q & 1)
#pragma unroll
            for (int sl = 0; sl < 2; ++sl)
#pragma unroll
                for (int nb = 0; nb < NB; ++nb)
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const uint32_t ra = red + (uint32_t)(((sl * NB + nb) * 4 + q) * 128);
                        tot[sl][nb][q] = ((tot[sl][nb][q] + sm_lds32(ra)) + sm_lds32(ra + red_group)) + sm_lds32(ra + 2 * red_group);
                    }
            if (whole) {
#pragma unroll
                for (int sl = 0; sl < 2; ++sl) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int gn = n0 + rows[sl][h];
                        const float bv = (bias != nullptr && gn < p.N) ? T::to_float(bias[gn]) : 0.0f;
#pragma unroll
                        for (int nb = 0; nb < NB; ++nb)
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const int m = 8 * nb + 2 * tig + e;
                                if (m < p.M && gn < p.N) {
                                    const ACT v = T::from_float(tot[sl][nb][2 * h + e] + bv);
                                    for (int o = 0; o < p.n_out; ++o)
                                        static_cast<ACT*>(p.y[o])[(int64_t)m * p.ldy + p.col0 + gn] = v;
                                }
                            }
                    }
                }
            } else {
                // this CTA's partial slot for the tile: 0 if it is the first tile the CTA touches, else 1;
                // layout [m][128 features]
                const int which = (tile == tile0) ? 0 : 1;
                float* mine = partial + ((size_t)cta * 2 + which) * (size_t)(kSmRows * p.m_pad);
#pragma unroll
                for (int sl = 0; sl < 2; ++sl)
#pragma unroll
                    for (int nb = 0; nb < NB; ++nb)
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            __stcg(mine + (8 * nb + 2 * tig + (q & 1)) * kSmRows + rows[sl][q >> 1], tot[sl][nb][q]);
                if (!final_seg && s1 != S) {
                    // a contributor segment with more work behind it: the publisher warp releases it
                    __syncwarp();
                    asm volatile("bar.arrive 2, 160;" ::: "memory");
                }
            }
        }
#pragma unroll
        for (int sl = 0; sl < 2; ++sl)
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) { tot[sl][nb][0] = tot[sl][nb][1] = tot[sl][nb][2] = tot[sl][nb][3] = 0.0f; }
        if (!whole && s1 == S) red_tile = tile;          // this CTA reduces the tile once its stream has ended
        if (tid == 0) SM_TRACE(30);
        sm_cons_sync();
        if (tid == 0) SM_TRACE(31);                                  // red is reused by the next segment; the partial stores are done
        if (!whole && final_seg && s1 != S && tid == 0) sm_contribute(counters, tile);
    }
    if (tid == 0) SM_TRACE(7);
    if (red_tile >= 0) {
        // ===== reducer duty: the other contributors' partials (lower CTA indices) =====
        const unsigned int tu0 = (unsigned int)red_tile * (unsigned int)S;
        const int c_first = sm_cta_of_unit(tu0, p), c_last = (int)cta;
        if (tid == 0) sm_await_contributors(counters, red_tile, c_last - c_first);
        sm_cons_sync();
        if (tid == 0) SM_TRACE(36);
        sm_fixup<ACT>(p, bias, partial, red_tile, c_first, c_last, tid, kSmConsThreads);
    }
    if (p.sync_world > 0) {
        // ===== cross-GPU completion (column-parallel layers): see PeerSync =====
        sm_cons_sync();                                      // every global store of this CTA has been issued
        if (warp == 0) {
            unsigned int last = 0u, epoch = 0u;
            if (lane == 0) {
                __threadfence_system();                      // ... and is performed, on the peers too, before the count moves
                const unsigned int old = atomicAdd(counters + kSmDoneIdx, 1u);
                if (old == gridDim.x - 1u) {
                    last = 1u;
                    counters[kSmDoneIdx] = 0u;               // clean for the next call
                    epoch = *p.sync_epoch + 1u;              // only this thread of this grid touches the counter
                    *p.sync_epoch = epoch;
                }
            }
            last = __shfl_sync(0xffffffffu, last, 0);
            epoch = __shfl_sync(0xffffffffu, epoch, 0);
            if (last) {
                // one lane per peer: all signals leave together and all peers are polled together (one NVLink round trip
                // instead of world - 1 of them)
                __threadfence_system();                      // the other CTAs' stores (observed through the counter) come first
                if (lane < p.sync_world && lane != p.sync_rank) {
                    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.sync_flags[lane] + p.sync_rank), "r"(epoch) : "memory");
                    unsigned int seen = 0, spins = 0;
                    for (;;) {
                        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(p.sync_flags[p.sync_rank] + lane) : "memory");
                        if ((int)(seen - epoch) >= 0 || ++spins > (1u << 28)) break;
                    }
                }
                __syncwarp();
            }
        }
    }
#ifdef QUANTA_SMALL_TRACE
    if (tid == 0) {
        SM_TRACE(37);
        unsigned long long g; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g)); g_sm_trace[blockIdx.x][39] = (long long)g;
    }
#endif
}

#ifdef QUANTA_SMALL_TRACE
extern "C" __attribute__((visibility("default"))) int quanta_debug_small_trace(long long* host_out) {
    return (int)cudaMemcpyFromSymbol(host_out, g_sm_trace, sizeof(long long) * kNumSMs * 40);
}
#endif

// ---- host side --------------------------------------------------------------

// The small-batch kernel serves M <= 16 with blockwise-64 parameters on K % 256 == 0.
bool gemm_small_eligible(int64_t M, int64_t N, int64_t K, int64_t block, const void* scale, const void* zp) {
    if (M > kSmMaxM || block != 64 || (K % kSmKGran) != 0) return false;
    if ((reinterpret_cast<uintptr_t>(scale) | reinterpret_cast<uintptr_t>(zp)) & 15) return false;
    const int64_t n_tiles = (N + kSmRows - 1) / kSmRows;
    if (n_tiles > kSmCounterBytes / 4) return false;
    const unsigned long long steps = (unsigned long long)(K / kSmKGran);       // >= S for both code widths
    if ((unsigned long long)n_tiles * steps * (unsigned long long)(kNumSMs + 1) >= (1ull << 32)) return false;
    if ((unsigned long long)n_tiles * steps * steps >= (1ull << 32)) return false;   // the division-free u / S (SmallParams::s_magic)
    return true;
}

template <typename ACT, int BITS, int NB, bool NF4, int XW>
static int gemm_small_launch_nb(const ACT* x, const uint8_t* wq, const float* scale, const float* zp, const ACT* bias,
                                void* const* ys, int n_out, int64_t ldy, int64_t col0, int64_t M, int64_t N, int64_t K,
                                void* workspace, size_t ws_bytes, cudaStream_t st, const PeerSync* sync) {
    SmallParams p;
    p.sync_world = 0; p.sync_rank = 0; p.sync_epoch = nullptr;
    for (int o = 0; o < kSmMaxOut; ++o) p.sync_flags[o] = nullptr;
    if (sync) {
        if (sync->world < 2 || sync->world > kSmMaxOut || sync->rank < 0 || sync->rank >= sync->world) return QUANTA_EINVAL;
        if ((N + kSmRows - 1) / kSmRows >= kSmDoneIdx) return QUANTA_EUNSUPPORTED;
        if (!sync->epoch_counter) return QUANTA_EINVAL;
        p.sync_world = sync->world; p.sync_rank = sync->rank; p.sync_epoch = sync->epoch_counter;
        for (int r = 0; r < sync->world; ++r) {
            if (!sync->flags[r]) return QUANTA_EINVAL;
            p.sync_flags[r] = static_cast<unsigned int*>(sync->flags[r]);
        }
    }
    p.M = (int)M; p.N = (int)N; p.K = (int)K;
    p.m_pad = 8 * NB;
    p.n_tiles = (int)((N + kSmRows - 1) / kSmRows);
    using G = SmGeom<BITS, NF4>;
    if (reinterpret_cast<uintptr_t>(x) & 15) return QUANTA_EINVAL;          // 16-byte activation loads
    p.S = (int)((K + G::kStepK - 1) / G::kStepK);
    p.U = (unsigned int)p.n_tiles * (unsigned int)p.S;
    const int sms = device_sm_count();
    // How many CTAs.  An even cut of the unit range over all SMs streams for the shortest time but ends on the
    // stream-K hand-over (partial stores, release, acquire, fix-up: ~2.5 stage times at M <= 8, more for wider partials)
    // and gives most CTAs two segments; k CTAs per row tile (k = 1: whole tiles, no hand-over at all) stream longer and
    // finish sooner when the tile count is close to a divisor of the SM count.  Costs in stage times, fitted to
    // 4096 x 14336 (32 tiles) and 14336 x 4096 (112 tiles: 11.3 us with one CTA per tile, 12.3 us with 148 ranges).
    int n_cta = (int)(p.U < (unsigned int)sms ? p.U : (unsigned int)sms);
    if (p.n_tiles <= sms) {
        // Costs of the two endings in stage times, fitted to measurements (W4, stage = 0.9 us at M <= 8, 1.3 us above):
        // an even cut ends on the hand-over AND gives most CTAs two segments; k CTAs per tile end on the hand-over only
        // (k > 1) or on nothing (k = 1).  They are fixed times, so they shrink in stage units as the stage grows (8-bit).
        const double f = BITS == 8 ? 2.0 / 3.0 : 1.0;
        // (M <= 8: k > 1 measured 0.2-0.5 us slower than the even cut wherever the two were close, hence 3.0)
        const double h_even = f * (NB == 1 ? 3.05 : 2.3), h_tile = f * (NB == 1 ? 3.0 : 0.85);
        double best = (double)p.U / n_cta + h_even;
        for (int k = 1; k * p.n_tiles <= sms && k <= p.S; ++k) {
            const double cost = (double)((p.S + k - 1) / k) + (k > 1 ? h_tile : 0.0);
            if (cost <= best && p.S % k == 0) { best = cost; n_cta = k * p.n_tiles; }
        }
    }
    p.G = n_cta;
    p.q = p.U / (unsigned int)p.G;
    p.r = p.U % (unsigned int)p.G;
    // u / S as a multiplication: exact for u <= U because U * (magic * S - 2^32) < U * S < 2^32 (gemm_small_eligible)
    p.s_magic = p.S == 1 ? 0u : (unsigned int)(((1ull << 32) + (unsigned long long)p.S - 1ull) / (unsigned long long)p.S);
    p.x_slot_bytes = (uint32_t)(NB * G::kBlk * (1024 + 32));
    const uint32_t red_bytes = (uint32_t)(3 * 4 * 2 * NB * 4 * 128);
    const uint32_t bar_bytes = 256;
    const uint32_t budget = 226u * 1024u;
    // The activation ring is sized first — 4 slots for M <= 8, 3 for M > 8 (measured at 4096 x 14336, M = 16: 3 slots +
    // 3 stages 17.0 us, 2 + 4: 19.3, 4 + 3: 18.4; its staging warps prefetch only one unit in registers there) — and
    // the weight ring gets what is left.
    const int xring = NB == 1 ? kSmMaxXRing : 3;
    const uint32_t lut_bytes = NF4 ? kSmLutBytes : 0u;
    int ring = (int)((budget - (uint32_t)xring * p.x_slot_bytes - red_bytes - bar_bytes - lut_bytes) / G::kStageBytes);
    if (ring > kSmMaxRing) ring = kSmMaxRing;
    if (ring < 2) return QUANTA_EUNSUPPORTED;
    p.R = ring;
    p.XR = xring;
    p.window = kSmStartWindow < ring ? kSmStartWindow : ring;
    const uint32_t x_bytes = (uint32_t)xring * p.x_slot_bytes;
    p.x_off = (uint32_t)ring * G::kStageBytes;
    p.lut_off = p.x_off + x_bytes;
    p.red_off = p.lut_off + lut_bytes;
    p.bar_off = p.red_off + red_bytes;
    const int smem = (int)(p.bar_off + bar_bytes);
    p.ldy = (int)ldy; p.col0 = (int)col0; p.n_out = n_out;
    bool aligned8 = true;
    for (int o = 0; o < kSmMaxOut; ++o) {
        p.y[o] = o < n_out ? ys[o] : nullptr;
        if (o < n_out) aligned8 = aligned8 && (reinterpret_cast<uintptr_t>(ys[o]) & 7) == 0;
    }
    p.vec_y = (aligned8 && (ldy & 3) == 0 && (col0 & 3) == 0) ? 1 : 0;

    const size_t need = (size_t)kSmCounterBytes + (size_t)p.G * 2 * kSmRows * (size_t)p.m_pad * sizeof(float) + 256;
    if (!workspace || ws_bytes < need) return QUANTA_EWORKSPACE;
    uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    unsigned int* counters = reinterpret_cast<unsigned int*>(ws);
    float* partial = reinterpret_cast<float*>(ws + kSmCounterBytes);

    CUtensorMap tmap_w, tmap_s, tmap_z;
    const uint64_t wrow_bytes = (uint64_t)K * BITS / 8;
    int rc = make_tensor_map_2d(&tmap_w, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, wq, wrow_bytes, (uint64_t)N, wrow_bytes, 128,
                                kSmRows, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    const uint64_t sstride = (uint64_t)(K / 64);
    rc = make_tensor_map_2d(&tmap_s, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, scale, sstride, (uint64_t)N, sstride * 4, G::kBlk, kSmRows,
                            CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
    rc = make_tensor_map_2d(&tmap_z, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, zp, sstride, (uint64_t)N, sstride * 4, G::kBlk, kSmRows,
                            CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;

    auto kern = gemm_small_kernel<ACT, BITS, NB, NF4, XW>;
    if (int e = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), smem)) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)p.G);
    cfg.blockDim = dim3(sm_threads(XW));
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tmap_w, tmap_s, tmap_z, x, bias, counters, partial, p);
    return cuda_status(e != cudaSuccess ? e : cudaGetLastError());
}

template <typename ACT, int BITS>
int gemm_small_launch(const ACT* x, const uint8_t* wq, const float* scale, const float* zp, const ACT* bias, void* const* ys,
                      int n_out, int64_t ldy, int64_t col0, int64_t M, int64_t N, int64_t K, void* workspace, size_t ws_bytes,
                      cudaStream_t st, int nf4, const PeerSync* sync) {
    const bool one = M == 1;                                 // a single batch row: two staging warps (see sm_threads)
    if (nf4) {
        // 4-bit codes index the NF4 table, `scale` holds abs_max per block, `zp` is not read
        if (BITS != 4) return QUANTA_EINVAL;
        if (one) return gemm_small_launch_nb<ACT, 4, 1, true, 2>(x, wq, scale, zp, bias, ys, n_out, ldy, col0, M, N, K, workspace, ws_bytes, st, sync);
        if (M <= 8) return gemm_small_launch_nb<ACT, 4, 1, true, 4>(x, wq, scale, zp, bias, ys, n_out, ldy, col0, M, N, K, workspace, ws_bytes, st, sync);
        return gemm_small_launch_nb<ACT, 4, 2, true, 4>(x, wq, scale, zp, bias, ys, n_out, ldy, col0, M, N, K, workspace, ws_bytes, st, sync);
    }
    if (one) return gemm_small_launch_nb<ACT, BITS, 1, false, 2>(x, wq, scale, zp, bias, ys, n_out, ldy, col0, M, N, K, workspace, ws_bytes, st, sync);
    if (M <= 8) return gemm_small_launch_nb<ACT, BITS, 1, false, 4>(x, wq, scale, zp, bias, ys, n_out, ldy, col0, M, N, K, workspace, ws_bytes, st, sync);
    return gemm_small_launch_nb<ACT, BITS, 2, false, 4>(x, wq, scale, zp, bias, ys, n_out, ldy, col0, M, N, K, workspace, ws_bytes, st, sync);
}

#define QUANTA_SMALL_INST(ACT, BITS)                                                                                    \
    template int gemm_small_launch<ACT, BITS>(const ACT*, const uint8_t*, const float*, const float*, const ACT*, void* const*, \
                                              int, int64_t, int64_t, int64_t, int64_t, int64_t, void*, size_t, cudaStream_t, int, \
                                              const PeerSync*);
QUANTA_SMALL_INST(__nv_bfloat16, 4)
QUANTA_SMALL_INST(__nv_bfloat16, 8)
QUANTA_SMALL_INST(__half, 4)
QUANTA_SMALL_INST(__half, 8)

}  // namespace quanta
