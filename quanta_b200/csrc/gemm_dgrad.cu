// Input gradient of the quantized linear layers on the 5th-generation tensor cores:
//     dx[M,K] = dy[M,N] . dequant(Wq)[N,K]
// The weight is frozen, so this is the only gradient the layers need.  Weight formats: blockwise
// affine 4/8-bit and NF4 (Linear4bit, Linear8bitLt), and the int8 row-wise codes of the outlier
// split (ROW8: W16[n,k] = round_act(qw[n,k] / cw[n]), the 16-bit weights of outlier.cu's outlier
// columns; the straight-through gradient of the LLM.int8() product).  It is the forward GEMM
// (gemm.cu) with the weight used the other way round: the reduction runs over N (out_features)
// and the output features are K (in_features).
//
// Mapping (swap-AB as in the forward): 128 output features k of a tile are the UMMA M dimension
// (one TMEM lane each), the batch rows are the UMMA N dimension (16..256):
//     D[k, m] (fp32, TMEM) += A[k, n] (dequantized W^T, smem) * B[m, n] (dy, smem)
// A stored code row n is contiguous in k, i.e. along the MMA's M dimension, so the dequantized
// weights form an MN-major A operand.  They are written to shared memory in the MN-major
// SWIZZLE_128B layout and the MMA reads A from there (tcgen05.mma ... a-desc, b-desc with the
// A-major bit set).  A TMEM A operand is K-major per lane and does not fit this orientation.
//
// Persistent, warp-specialised CTA (one per SM), 24 warps:
//   warp 0      TMA ring of raw weight codes: stages of [256 code rows x 128 k] (64 B per row at
//               4 bits, unswizzled; 128 B at 8 bits, SWIZZLE_128B); rows past N arrive zero-filled
//   warp 1      TMA ring of dy tiles [mb x 64 n] (SWIZZLE_128B, K-major B operand, as x in the forward)
//   warp 2      TMEM allocation; one lane issues tcgen05.mma.kind::f16 (4 x K=16 per 64-n block)
//   warps 4-7   epilogue (the forward's, without the bias): TMEM lane = output column k
//   warps 8-23  dequantize: 2 groups x 8 warps; group g owns the 64-n blocks g and g + 2 of every
//               stage (A slots g and g + 2).  Thread -> (code row, quarter of the 128 k): 32 codes
//               -> 32 16-bit weights with the forward's dequant_word4 / dequant_word8 / NF4 table
//               (ROW8: dequant_word8_row) -> four 16-byte shared-memory stores into the A slot
// Work is split stream-K style over (k tile, n stage) units, with the forward's deterministic
// fix-up, counters and workspace (GemmParams in the OUTPUT's terms: p.N = in_features K is the
// output width, p.K = out_features N is the reduction length).
//
// Tile width: 128 k per tile.  A 256-k tile would read 128-byte instead of 64-byte row pieces at
// 4 bits, but needs two accumulators per buffer (mb = 256 then fills TMEM with one buffer) and
// 128 KB of A slots per stage; DESIGN §4.1c has the measured rates of the 128-k tile.
#include "gemm_tc.cuh"

namespace quanta {

constexpr int kDgCtrlWarps = 4, kDgEpiWarps = 4, kDgGroups = 2, kDgGroupWarps = 8;
constexpr int kDgDqWarps = kDgGroups * kDgGroupWarps;
constexpr int kDgFirstEpiWarp = kDgCtrlWarps, kDgFirstDqWarp = kDgCtrlWarps + kDgEpiWarps;
constexpr int kDgThreads = 32 * (kDgCtrlWarps + kDgEpiWarps + kDgDqWarps);
constexpr int kDgRows = kKbPerStage * kBlockK;            // code rows (reduction values) per raw stage
constexpr uint32_t kASlotBytes = kTileN * kBlockK * 2;    // one 64-n block of W^T in 16 bits
constexpr uint32_t kAMnBlockBytes = kASlotBytes / 2;      // 64 k x 64 n: one MN block of the slot
constexpr int kASlotsDg = kKbPerStage;                    // A slot j <-> 64-n block j of every stage

// MN-major, SWIZZLE_128B shared-memory matrix descriptor.  Swizzle atom: 8 n rows of 128 bytes =
// 64 k values each; atoms along n are 1024 bytes apart (SBO), the second 64 k of the 128-k tile
// starts kAMnBlockBytes later (LBO).  Descriptor version 1 (sm_100).
__device__ __forceinline__ uint64_t smem_desc_mn_sw128(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(kAMnBlockBytes >> 4) << 16) |
           ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// D[tmem] (+)= A[smem descriptor] * B[smem descriptor]
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// int8 row-wise codes (rowwise_quantize_sym): four signed codes -> round_act(q / cw), bit for bit the
// forward's round_act(__fdiv_rn(q, cw)).  XOR 0x80 makes each byte q + 128, which PRMT drops into
// 0x4700uu00 = 32768 + q + 128; one add leaves q exactly.  With y = RN(1/cw) hoisted per row,
// q0 = q y; r = fma(-cw, q0, q); fma(y, r, q0) is the correctly rounded quotient for every code and
// every cw in [2^-60, 2^60] (affine_quotient's window; exhaustive check: tools/check_rowwise_div.c).
// Rows outside the window (cw = inf for an all-zero or subnormal row, cw < 2^-60 for a huge one)
// are redone by dequant_word8_row_div.  Pairs of lanes run as f32x2 FADD2 / FMUL2 / FFMA2.
__device__ __forceinline__ float2 codes8_row(uint32_t u, int e) {
    const float2 f = make_float2(__uint_as_float(prmt_(u, 0x47000000u, 0x7504u | ((2 * e) << 4))),
                                 __uint_as_float(prmt_(u, 0x47000000u, 0x7504u | ((2 * e + 1) << 4))));
    return __fadd2_rn(f, make_float2(-32896.0f, -32896.0f));
}
template <typename ACT>
__device__ __forceinline__ void dequant_word8_row(uint32_t w, float2 ncw2, float2 y2, uint32_t* out) {
    const uint32_t u = w ^ 0x80808080u;
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const float2 a = codes8_row(u, e);
        const float2 q0 = __fmul2_rn(a, y2);
        const float2 q = __ffma2_rn(y2, __ffma2_rn(ncw2, q0, a), q0);
        out[e] = ActTraits<ACT>::pack(q.x, q.y);
    }
}
template <typename ACT>
__device__ __forceinline__ void dequant_word8_row_div(uint32_t w, float cw, uint32_t* out) {
    const uint32_t u = w ^ 0x80808080u;
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const float2 a = codes8_row(u, e);
        out[e] = ActTraits<ACT>::pack(__fdiv_rn(a.x, cw), __fdiv_rn(a.y, cw));
    }
}

template <typename ACT, int BITS, bool ROW8>
__global__ void __launch_bounds__(kDgThreads, 1)
gemm_dgrad_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_dy,
                  const __grid_constant__ GemmOutputs<1> outs, const float* __restrict__ scale, const float* __restrict__ zp,
                  unsigned int* __restrict__ counters, float* __restrict__ partial, const __grid_constant__ GemmParams p) {
    using AT = ActTraits<ACT>;
    constexpr uint32_t kRowBytes = kTileN * BITS / 8;          // one code row of a k tile
    constexpr uint32_t kRawBytes = kRowBytes * kDgRows;
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t raw_full[kMaxRing], raw_empty[kMaxRing], x_full[kMaxRing], x_empty[kMaxRing];
    __shared__ uint64_t a_full[kASlotsDg], a_empty[kASlotsDg], d_full[2], d_empty[2];
    __shared__ uint32_t tmem_base_slot;
    __shared__ int fix_flag;
    __shared__ int fin_tile;
    __shared__ __align__(1024) float stage[16][kTileN];        // epilogue transpose buffer (8 KB)
    __shared__ uint32_t nf4_pairs[256];

    // shared memory: [A slots: 4 x 16 KB][raw ring: raw_stages x 16|32 KB][dy ring: x_stages x mb x 128 B]
    const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const unsigned int cta = blockIdx.x;
    auto a_addr = [&](int j) { return smem + (uint32_t)j * kASlotBytes; };
    auto r_addr = [&](int s) { return smem + kASlotsDg * kASlotBytes + (uint32_t)s * kRawBytes; };
    auto x_addr = [&](int s) { return smem + p.x_ring_off + (uint32_t)s * p.x_slot_bytes; };

    SegWalk walk;
    walk.init(p, cta);
    int tile, s0, s1;
    if (tid == 32 * kDgFirstEpiWarp) fin_tile = -1;
    if (BITS == 4 && p.nf4 && tid >= 32 * kDgFirstDqWarp && tid < 32 * kDgFirstDqWarp + 256) {
        const int b = tid - 32 * kDgFirstDqWarp;
        nf4_pairs[b] = AT::pack(kNf4Levels[b & 15], kNf4Levels[b >> 4]);
    }

    // PDL as in the forward: release dependents at once; the weight stream (codes, scales) starts
    // at once; dy loads and every global write wait for the previous kernel.  dx is never a weight,
    // so the early release is sound (common.cuh).
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (warp == 0) {
        // ===== raw weight codes =====
        if (lane == 0) {
            for (int s = 0; s < p.raw_stages; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], kDgDqWarps); }
            fence_barrier_init();
            prefetch_tensormap(&tmap_w);
        }
        __syncwarp();
        asm volatile("barrier.arrive 2, %0;" ::"n"(kDgThreads) : "memory");
        const uint64_t pol_w = policy_evict_first();
        int slot = 0, issued = 0;
        uint32_t ph = 0;
        while (walk.next(tile, s0, s1)) {
            int k_idx, m_idx;
            split_tile(tile, p, k_idx, m_idx);
            for (int s = s0; s < s1; ++s) {
                if (issued >= p.raw_stages) mbar_wait(&raw_empty[slot], ph ^ 1);
                if (elect_one()) {
                    mbar_arrive_expect_tx(&raw_full[slot], kRawBytes);
                    tma_load_2d_plain(r_addr(slot), &tmap_w, smem_u32(&raw_full[slot]), k_idx * (int)kRowBytes, s * kDgRows, pol_w);
                }
                __syncwarp();
                ++issued;
                if (++slot == p.raw_stages) { slot = 0; ph ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===== dy tiles: one 64-n block per slot =====
        if (lane == 0) {
            for (int s = 0; s < p.x_stages; ++s) { mbar_init(&x_full[s], 1); mbar_init(&x_empty[s], 1); }
            fence_barrier_init();
            prefetch_tensormap(&tmap_dy);
        }
        __syncwarp();
        asm volatile("barrier.arrive 2, %0;" ::"n"(kDgThreads) : "memory");
        const uint64_t pol_x = policy_evict_last();          // dy is re-read by every k tile
        asm volatile("griddepcontrol.wait;" ::: "memory");
        int slot = 0, issued = 0;
        uint32_t ph = 0;
        while (walk.next(tile, s0, s1)) {
            int k_idx, m_idx;
            split_tile(tile, p, k_idx, m_idx);
            const int m0 = m_idx * p.mb;
            for (int s = s0; s < s1; ++s) {
                for (int j = 0; j < kKbPerStage; ++j) {
                    if (issued >= p.x_stages) mbar_wait(&x_empty[slot], ph ^ 1);
                    if (elect_one()) {
                        mbar_arrive_expect_tx(&x_full[slot], p.x_slot_bytes);
                        // columns past N arrive zero-filled
                        tma_load_2d_plain(x_addr(slot), &tmap_dy, smem_u32(&x_full[slot]), (s * kKbPerStage + j) * kBlockK, m0, pol_x);
                    }
                    __syncwarp();
                    ++issued;
                    if (++slot == p.x_stages) { slot = 0; ph ^= 1; }
                }
            }
        }
    } else {
        if (warp == 2) {
            tmem_alloc(smem_u32(&tmem_base_slot), kTmemCols);
        } else if (warp == 3 && lane == 0) {
            for (int s = 0; s < kASlotsDg; ++s) { mbar_init(&a_full[s], kDgGroupWarps); mbar_init(&a_empty[s], 1); }
            for (int s = 0; s < 2; ++s) { mbar_init(&d_full[s], 1); mbar_init(&d_empty[s], kDgEpiWarps); }
            fence_barrier_init();
        }
        __syncwarp();
        tc_fence_before();
        asm volatile("barrier.sync 2, %0;" ::"n"(kDgThreads) : "memory");
    }
    tc_fence_after();
    const uint32_t tmem = tmem_base_slot;

    if (warp == 2) {
        // ===== MMA issuer =====
        const uint32_t idesc = (1u << 4) | (AT::kFmt << 7) | (AT::kFmt << 10) | (1u << 15) /* A MN-major */ |
                               ((uint32_t)(p.mb >> 3) << 17) | ((uint32_t)(kTileN >> 4) << 24);
        const uint32_t nacc = (uint32_t)p.nacc;
        int sx = 0, seg = 0, sc = 0;
        uint32_t px = 0;
        while (walk.next(tile, s0, s1)) {
            const int buf = seg & 1;
            const uint32_t use = (uint32_t)(seg >> 1);
            mbar_wait(&d_empty[buf], (use & 1) ^ 1);
            const uint32_t tmem_d = tmem + (uint32_t)(buf * p.nacc * p.mb);
            uint32_t touched = 0;
            for (int s = s0; s < s1; ++s, ++sc) {
                const int nkb = min(kKbPerStage, p.total_kb - s * kKbPerStage);
#pragma unroll
                for (int j = 0; j < kKbPerStage; ++j) {
                    mbar_wait(&a_full[j], (uint32_t)sc & 1u);       // block j of the stage is in its A slot
                    mbar_wait(&x_full[sx], px);
                    tc_fence_after();
                    const bool live = j < nkb;
                    uint32_t acc_idx[4], acc_flag[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        acc_idx[k] = (uint32_t)(4 * j + k) & (nacc - 1u);
                        acc_flag[k] = (touched >> acc_idx[k]) & 1u;
                        if (live) touched |= 1u << acc_idx[k];
                    }
                    if (elect_one()) {
                        if (live) {
                            const uint64_t da = smem_desc_mn_sw128(a_addr(j));
                            const uint64_t db = smem_desc_sw128(x_addr(sx));
#pragma unroll
                            for (int k = 0; k < kBlockK / 16; ++k)    // 16 n per MMA: two swizzle atoms of A, 32 bytes of B
                                umma_f16_ss(tmem_d + acc_idx[k] * (uint32_t)p.mb, da + (uint64_t)(k * (2048 >> 4)), db + 2 * k,
                                            idesc, acc_flag[k]);
                        }
                        umma_commit(&x_empty[sx]);
                        umma_commit(&a_empty[j]);
                    }
                    __syncwarp();
                    if (++sx == p.x_stages) { sx = 0; px ^= 1; }
                }
            }
            if (elect_one()) umma_commit(&d_full[buf]);
            __syncwarp();
            ++seg;
        }
    } else if (warp >= kDgFirstEpiWarp && warp < kDgFirstDqWarp) {
        // ===== epilogue: TMEM lane = output column k =====
        asm volatile("griddepcontrol.wait;" ::: "memory");
        const int quarter = warp & 3;
        const int row = 32 * quarter + lane;
        const int etid = tid - 32 * kDgFirstEpiWarp;
        if (etid == 0 && p.y_tma) prefetch_tensormap(&outs.maps[0]);
        int seg = 0;
        while (walk.next(tile, s0, s1)) {
            const int buf = seg & 1;
            const uint32_t use = (uint32_t)(seg >> 1);
            int k_tile, m_tile;
            split_tile(tile, p, k_tile, m_tile);
            const int m0 = m_tile * p.mb;
            const int m_valid = min(p.mb, p.M - m0);
            const bool whole = (s0 == 0 && s1 == p.S);
            const bool last_seg = walk.u >= walk.u1;
            const int which = (tile == tile_of_unit(first_unit(cta, p), p)) ? 0 : 1;
            float* mine = partial + ((size_t)cta * 2 + which) * (size_t)(kTileN * p.mb);

            mbar_wait(&d_full[buf], use & 1);
            tc_fence_after();
            const uint32_t taddr = tmem + ((uint32_t)(32 * quarter) << 16) + (uint32_t)(buf * p.nacc * p.mb);
            const int f4 = 4 * (etid & 31);
            const int gk4 = k_tile * kTileN + f4;
            const bool vec_ok = p.vec_store && gk4 + 3 < p.N;
            const int last_nkb = (s1 == p.S) ? p.total_kb - (p.S - 1) * kKbPerStage : kKbPerStage;
            const int nv = min(p.nacc, 4 * ((s1 - s0 - 1) * kKbPerStage + last_nkb));
            for (int c0 = 0; c0 < p.mb; c0 += 16) {
                uint32_t r[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) r[j] = 0u;
                for (int a = 0; a < nv; ++a) {
                    uint32_t t[16];
                    tmem_ld16(taddr + (uint32_t)(a * p.mb) + c0, t);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(t[j]));
                }
                if (whole && p.y_tma) {
                    // whole tile: [16 rows x 128 columns] staged in shared memory, one TMA store per chunk
                    ACT* sbuf = reinterpret_cast<ACT*>(&stage[0][0]) + ((c0 >> 4) & 1) * (16 * kTileN);
                    if (etid == 0 && c0 >= 32) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                    asm volatile("bar.sync 1, %0;" ::"n"(32 * kDgEpiWarps) : "memory");
#pragma unroll
                    for (int j = 0; j < 16; ++j) sbuf[j * kTileN + row] = AT::from_float(__uint_as_float(r[j]));
                    fence_proxy_async_smem();
                    asm volatile("bar.sync 1, %0;" ::"n"(32 * kDgEpiWarps) : "memory");
                    if (etid == 0 && c0 < m_valid) {
                        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                                     ::"l"(reinterpret_cast<uint64_t>(&outs.maps[0])), "r"(smem_u32(sbuf)),
                                       "r"(k_tile * kTileN), "r"(m0 + c0) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    continue;
                }
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kDgEpiWarps) : "memory");
#pragma unroll
                for (int j = 0; j < 16; ++j) stage[j][row] = __uint_as_float(r[j]);
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kDgEpiWarps) : "memory");
                if (c0 < m_valid) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int ml = 4 * q + (etid >> 5);
                        const int m = c0 + ml;
                        if (m < m_valid) {
                            const float4 v = *reinterpret_cast<const float4*>(&stage[ml][f4]);
                            if (whole) {
                                ACT* dst = static_cast<ACT*>(outs.y[0]) + (int64_t)(m0 + m) * p.ldy + gk4;
                                if (vec_ok) {
                                    uint2 pk;
                                    pk.x = AT::pack(v.x, v.y);
                                    pk.y = AT::pack(v.z, v.w);
                                    *reinterpret_cast<uint2*>(dst) = pk;
                                } else {
                                    const float o[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                                    for (int e = 0; e < 4; ++e) if (gk4 + e < p.N) dst[e] = AT::from_float(o[e]);
                                }
                            } else {
                                *reinterpret_cast<float4*>(mine + m * kTileN + f4) = v;
                            }
                        }
                    }
                }
            }
            if (whole && p.y_tma && etid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&d_empty[buf]);
            if (!whole) {
                // stream-K fix-up exactly as in the forward: the last CTA to arrive reduces every partial
                const unsigned int tu0 = (unsigned int)tile * (unsigned int)p.S;
                const int c_first = cta_of_unit(tu0, p), c_last = cta_of_unit(tu0 + (unsigned int)p.S - 1u, p);
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kDgEpiWarps) : "memory");
                if (etid == 0) {
                    __threadfence();
                    const unsigned int old = atomicAdd(&counters[tile], 1u);
                    __threadfence();
                    const int last = (old == (unsigned int)(c_last - c_first)) ? 1 : 0;
                    if (last) counters[tile] = 0u;
                    fix_flag = last;
                }
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kDgEpiWarps) : "memory");
                if (fix_flag) {
                    if (last_seg && p.mb >= 64) {
                        if (etid == 0) fin_tile = tile;
                    } else {
                        fixup_reduce<ACT, 1>(p, outs, nullptr, partial, tile, etid, 32 * kDgEpiWarps);
                    }
                }
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kDgEpiWarps) : "memory");
            }
            ++seg;
        }
    } else if (warp >= kDgFirstDqWarp) {
        // ===== dequantize: thread = (code row of a 64-n block, quarter of the tile's 128 k) =====
        using V2 = typename AT::V2;
        const int group = (warp - kDgFirstDqWarp) / kDgGroupWarps;
        const int gt = (warp - kDgFirstDqWarp) % kDgGroupWarps * 32 + lane;
        const int rl = gt >> 2;                       // code row within the 64-n block
        const int q = gt & 3;                         // k values 32q .. 32q + 31 of the tile
        const uint32_t sw = (uint32_t)(rl & 7);
        // MN-major SWIZZLE_128B: element (k, n) of a slot at (k / 64) * LBO + (n / 8) * 1024 + (n % 8) * 128
        // + (((k % 64) / 8) ^ (n % 8)) * 16 + (k % 8) * 2; this thread's k / 64 is q / 2, its chunks 4 (q & 1) + i
        const uint32_t a_off = (uint32_t)(q >> 1) * kAMnBlockBytes + (uint32_t)(rl >> 3) * 1024u + sw * 128u;
        const V2 c2 = AT::dup(AT::kCentre);

        // scale / zero-point of this thread's two code rows: loaded one stage ahead
        SegWalk ahead = walk;
        int a_tile = 0, a_s = 0, a_s1 = 0;
        bool a_ok = ahead.next(a_tile, a_s, a_s1);
        float sv[2], zv[2];
        auto fetch_params = [&](int t, int s) {
            int k_idx, m_idx;
            split_tile(t, p, k_idx, m_idx);
            const int col = min((k_idx * kTileN + 32 * q) >> (6 + p.block_shift), p.scale_stride - 1);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int n = min(s * kDgRows + (group + 2 * h) * kBlockK + rl, p.K - 1);
                const int64_t i = (int64_t)n * p.scale_stride + col;
                sv[h] = __ldg(scale + i);
                zv[h] = (ROW8 || p.nf4) ? 0.0f : __ldg(zp + i);
            }
        };
        if (a_ok) fetch_params(a_tile, a_s);

        int sc = 0, rslot = 0;
        uint32_t rph = 0;
        while (walk.next(tile, s0, s1)) {
            for (int s = s0; s < s1; ++s, ++sc) {
                const int nkb = min(kKbPerStage, p.total_kb - s * kKbPerStage);
                const float cs[2] = {sv[0], sv[1]}, cz[2] = {zv[0], zv[1]};
                if (++a_s >= a_s1) a_ok = ahead.next(a_tile, a_s, a_s1);
                if (a_ok) fetch_params(a_tile, a_s);        // lands while this stage is processed
                mbar_wait(&raw_full[rslot], rph);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int j = group + 2 * h;
                    const int n = s * kDgRows + j * kBlockK + rl;
                    // the MMAs that read this A slot one stage ago are done
                    mbar_wait(&a_empty[j], ((uint32_t)sc & 1u) ^ 1u);
                    if (j < nkb) {
                        uint32_t out[16];
                        const uint32_t rrow = r_addr(rslot) + (uint32_t)(j * kBlockK + rl) * kRowBytes;
                        if (n >= p.K) {
#pragma unroll
                            for (int i = 0; i < 16; ++i) out[i] = 0u;     // rows past N (their codes are TMA zero fill)
                        } else if (BITS == 4 && p.nf4) {
                            const V2 s2 = AT::dup(cs[h]);
                            const uint4 rv = lds128g(rrow + (uint32_t)q * 16u);
                            const uint32_t w4[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    uint32_t pr = nf4_pairs[(w4[i] >> (8 * e)) & 0xFFu];
                                    V2 v = __hmul2(*reinterpret_cast<V2*>(&pr), s2);
                                    out[4 * i + e] = *reinterpret_cast<uint32_t*>(&v);
                                }
                            }
                        } else if (ROW8) {
                            // one multiplier per code row: scale_stride 1, so cs[h] = cw[n]
                            const float cw = cs[h], y = __frcp_rn(cw);
                            const float2 y2 = make_float2(y, y), ncw2 = make_float2(-cw, -cw);
#pragma unroll
                            for (int g = 0; g < 2; ++g) {
                                const uint4 rv = lds128g(rrow + (((uint32_t)(2 * q + g) ^ sw) << 4));
                                dequant_word8_row<ACT>(rv.x, ncw2, y2, out + 8 * g);
                                dequant_word8_row<ACT>(rv.y, ncw2, y2, out + 8 * g + 2);
                                dequant_word8_row<ACT>(rv.z, ncw2, y2, out + 8 * g + 4);
                                dequant_word8_row<ACT>(rv.w, ncw2, y2, out + 8 * g + 6);
                            }
                            if (!(cw >= 0x1p-60f && cw <= 0x1p60f)) {
#pragma unroll
                                for (int g = 0; g < 2; ++g) {
                                    const uint4 rv = lds128g(rrow + (((uint32_t)(2 * q + g) ^ sw) << 4));
                                    dequant_word8_row_div<ACT>(rv.x, cw, out + 8 * g);
                                    dequant_word8_row_div<ACT>(rv.y, cw, out + 8 * g + 2);
                                    dequant_word8_row_div<ACT>(rv.z, cw, out + 8 * g + 4);
                                    dequant_word8_row_div<ACT>(rv.w, cw, out + 8 * g + 6);
                                }
                            }
                        } else if (BITS == 4) {
                            const V2 s2 = AT::dup(cs[h]);
                            const V2 z2 = AT::dup(__fmaf_rn(8.0f, cs[h], cz[h]));
                            const uint4 rv = lds128g(rrow + (uint32_t)q * 16u);
                            dequant_word4<ACT>(rv.x, s2, z2, c2, out);
                            dequant_word4<ACT>(rv.y, s2, z2, c2, out + 4);
                            dequant_word4<ACT>(rv.z, s2, z2, c2, out + 8);
                            dequant_word4<ACT>(rv.w, s2, z2, c2, out + 12);
                        } else {
                            const float zc = __fmaf_rn(-32768.0f, cs[h], cz[h]);
#pragma unroll
                            for (int g = 0; g < 2; ++g) {
                                const uint4 rv = lds128g(rrow + (((uint32_t)(2 * q + g) ^ sw) << 4));
                                dequant_word8<ACT>(rv.x, cs[h], zc, out + 8 * g);
                                dequant_word8<ACT>(rv.y, cs[h], zc, out + 8 * g + 2);
                                dequant_word8<ACT>(rv.z, cs[h], zc, out + 8 * g + 4);
                                dequant_word8<ACT>(rv.w, cs[h], zc, out + 8 * g + 6);
                            }
                        }
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            sts128(a_addr(j) + a_off + ((((uint32_t)(4 * (q & 1) + i)) ^ sw) << 4),
                                   out[4 * i], out[4 * i + 1], out[4 * i + 2], out[4 * i + 3]);
                        fence_proxy_async_smem();              // generic-proxy stores -> tcgen05.mma reads
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&a_full[j]);
                }
                if (lane == 0) mbar_arrive(&raw_empty[rslot]);
                if (++rslot == p.raw_stages) { rslot = 0; rph ^= 1; }
            }
        }
    }

    if (warp >= kDgFirstEpiWarp && p.mb >= 64) {
        // a pending last-segment fix-up is reduced by the epilogue and dequant warps together
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("bar.sync 3, %0;" ::"n"(32 * (kDgEpiWarps + kDgDqWarps)) : "memory");
        const int ft = *reinterpret_cast<volatile int*>(&fin_tile);
        if (ft >= 0) fixup_reduce<ACT, 1>(p, outs, nullptr, partial, ft, tid - 32 * kDgFirstEpiWarp, 32 * (kDgEpiWarps + kDgDqWarps));
    }
    if (tid == 32 * kDgFirstEpiWarp) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem, kTmemCols); }
}

// ---- host side --------------------------------------------------------------

// ROW8: int8 row-wise codes, `scale` = cw [N], no zero-point, `block` unused
template <typename ACT, int BITS, bool ROW8 = false>
static int dgrad_launch(const ACT* dy, const uint8_t* wq, const float* scale, const float* zp, int64_t block, ACT* dx,
                        int64_t M, int64_t N, int64_t K, void* workspace, size_t ws_bytes, cudaStream_t st, int nf4) {
    constexpr uint32_t kRowBytes = kTileN * BITS / 8;
    constexpr uint32_t kRawBytes = kRowBytes * kDgRows;
    GemmParams p = {};
    p.M = (int)M; p.N = (int)K; p.K = (int)N;            // output [M, K], reduction over N
    int mb = (int)((M + 15) / 16 * 16);
    if (mb > 256) mb = 256;
    p.mb = mb;
    p.m_tiles = (int)((M + mb - 1) / mb);
    p.n_tiles = (int)((K + kTileN - 1) / kTileN);
    p.total_kb = (int)((N + kBlockK - 1) / kBlockK);
    p.S = (p.total_kb + kKbPerStage - 1) / kKbPerStage;
    p.nacc = mb <= 16 ? 8 : (mb <= 64 ? 4 : (mb <= 128 ? 2 : 1));     // 2 x nacc x mb <= 512 TMEM columns
    p.nbuf = 2;
    p.nf4 = nf4;
    p.n_out = 1; p.ldy = (int)K; p.col0 = 0;
    p.scale_stride = ROW8 ? 1 : (int)(K / block);
    int bs = 0; while (!ROW8 && (int64_t)(kBlockK << bs) < block) ++bs;
    p.block_shift = bs;
    p.vec4 = 0;

    const int tiles = p.n_tiles * p.m_tiles;
    if (tiles > kMaxTiles) return QUANTA_EUNSUPPORTED;
    if ((unsigned long long)tiles * (unsigned long long)p.S * (unsigned long long)(kNumSMs + 1) >= (1ull << 32)) return QUANTA_EUNSUPPORTED;
    p.U = (unsigned int)tiles * (unsigned int)p.S;
    p.G = choose_units(tiles, p.S, mb, (int)kRawBytes);
    p.uq = p.U / (unsigned int)p.G;
    p.ur = p.U % (unsigned int)p.G;
    {
        auto magic_for = [](unsigned int d, unsigned long long xmax, unsigned int* out) {
            if (d == 1) { *out = 0u; return true; }
            const unsigned long long m = ((1ull << 32) + d - 1ull) / d;
            *out = (unsigned int)m;
            return xmax * (m * d - (1ull << 32)) < (1ull << 32);
        };
        if (!magic_for((unsigned int)p.S, p.U, &p.s_magic) || !magic_for((unsigned int)p.n_tiles, (unsigned long long)tiles, &p.nt_magic))
            return QUANTA_EUNSUPPORTED;
    }
    p.x_kb_bytes = (uint32_t)mb * 128u;
    p.xkb = 1;
    p.x_slot_bytes = p.x_kb_bytes;
    p.raw_bytes = kRawBytes;
    // Shared memory: the A slots, a dy ring sized for the MMA, everything else for the raw-code ring.
    const uint32_t budget = 214u * 1024u;
    const uint32_t a_bytes = kASlotsDg * kASlotBytes;
    int x_stages = mb <= 64 ? 8 : (mb <= 128 ? 4 : (BITS == 4 ? 3 : 2));
    int raw_stages = (int)((budget - a_bytes - (uint32_t)x_stages * p.x_slot_bytes) / kRawBytes);
    if (raw_stages > kMaxRing) raw_stages = kMaxRing;
    if (raw_stages < 2) return QUANTA_EUNSUPPORTED;
    p.raw_stages = raw_stages;
    p.x_stages = x_stages;
    p.x_ring_off = a_bytes + (uint32_t)raw_stages * kRawBytes;

    const size_t need = (size_t)kCounterBytes + (size_t)p.G * 2 * kTileN * (size_t)mb * sizeof(float) + 256;
    if (!workspace || ws_bytes < need) return QUANTA_EWORKSPACE;
    uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    unsigned int* counters = reinterpret_cast<unsigned int*>(ws);
    float* partial = reinterpret_cast<float*>(ws + kCounterBytes);

    CUtensorMap tmap_w, tmap_dy;
    const uint64_t wrow_bytes = (uint64_t)K * BITS / 8;
    int rc = make_tensor_map_2d(&tmap_w, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, wq, wrow_bytes, (uint64_t)N, wrow_bytes, kRowBytes,
                                kDgRows, BITS == 4 ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    const uint64_t ld_dy = (uint64_t)(N + 7) / 8 * 8;       // row pitch of dy (include/quanta_b200.h)
    rc = make_tensor_map_2d(&tmap_dy, ActTraits<ACT>::kTma, 2, dy, (uint64_t)N, (uint64_t)M, ld_dy * 2, kBlockK, (uint32_t)mb,
                            CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    GemmOutputs<1> outs;
    outs.maps[0] = tmap_w;                                   // placeholder
    outs.y[0] = dx;
    p.vec_store = (reinterpret_cast<uintptr_t>(dx) & 7) == 0 ? 1 : 0;     // K % 16 == 0
    p.y_tma = (reinterpret_cast<uintptr_t>(dx) & 15) == 0 ? 1 : 0;
    if (p.y_tma) {
        rc = make_tensor_map_2d(&outs.maps[0], ActTraits<ACT>::kTma, 2, dx, (uint64_t)K, (uint64_t)M, (uint64_t)K * 2, kTileN, 16,
                                CU_TENSOR_MAP_SWIZZLE_NONE);
        if (rc) return rc;
    }
    auto kern = gemm_dgrad_kernel<ACT, BITS, ROW8>;
    const int smem = (int)(p.x_ring_off + (uint32_t)p.x_stages * p.x_slot_bytes + 1024);
    if (int e = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), smem)) return e;
    const cudaError_t e = launch_pdl(kern, dim3((unsigned)p.G), dim3(kDgThreads), (size_t)smem, st, tmap_w, tmap_dy, outs, scale, zp,
                                     counters, partial, p);
    return cuda_status(e != cudaSuccess ? e : cudaGetLastError());
}

// argument checks shared by every entry; all of them run before the first CUDA call.  fmt_ok: the
// entry's weight-format arguments are valid (QUANTA_EINVAL otherwise, like a null pointer).
static int dgrad_check(const void* dy, const void* wq, const float* scale, const void* dx, bool fmt_ok, int64_t M,
                       int64_t N, int64_t K) {
    if (!dy || !wq || !scale || !dx || M <= 0 || N <= 0 || K <= 0 || !fmt_ok) return QUANTA_EINVAL;
    if (M > INT32_MAX || N > INT32_MAX || K > INT32_MAX) return QUANTA_EUNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(wq)) & 15) return QUANTA_EUNSUPPORTED;
    return QUANTA_OK;
}
// blockwise formats: 4 or 8 bits, block = 64 * 2^j dividing K
static int dgrad_check_block(const void* dy, const uint8_t* wq, const float* scale, const void* dx, int bits,
                             int64_t block, int64_t M, int64_t N, int64_t K) {
    const bool fmt_ok = (bits == 4 || bits == 8) && block > 0 && block % kBlockK == 0 && K % block == 0;
    if (int rc = dgrad_check(dy, wq, scale, dx, fmt_ok, M, N, K)) return rc;
    return ((block / kBlockK) & (block / kBlockK - 1)) ? QUANTA_EUNSUPPORTED : QUANTA_OK;
}

}  // namespace quanta

using namespace quanta;

extern "C" int quanta_gemm_wna16_dgrad(const void* dy, int act_dtype, const uint8_t* wq, int bits, const float* scale,
                                       const float* zp, int64_t block, void* dx, int64_t M, int64_t N, int64_t K,
                                       void* workspace, size_t workspace_bytes, void* stream) {
    if (!zp) return QUANTA_EINVAL;
    if (int rc = dgrad_check_block(dy, wq, scale, dx, bits, block, M, N, K)) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (act_dtype == QUANTA_BF16) {
        using T = __nv_bfloat16;
        return bits == 4 ? dgrad_launch<T, 4>((const T*)dy, wq, scale, zp, block, (T*)dx, M, N, K, workspace, workspace_bytes, st, 0)
                         : dgrad_launch<T, 8>((const T*)dy, wq, scale, zp, block, (T*)dx, M, N, K, workspace, workspace_bytes, st, 0);
    }
    if (act_dtype == QUANTA_F16) {
        using T = __half;
        return bits == 4 ? dgrad_launch<T, 4>((const T*)dy, wq, scale, zp, block, (T*)dx, M, N, K, workspace, workspace_bytes, st, 0)
                         : dgrad_launch<T, 8>((const T*)dy, wq, scale, zp, block, (T*)dx, M, N, K, workspace, workspace_bytes, st, 0);
    }
    return QUANTA_EINVAL;
}

extern "C" int quanta_gemm_nf4a16_dgrad(const void* dy, int act_dtype, const uint8_t* wq, const float* absmax, int64_t block,
                                        void* dx, int64_t M, int64_t N, int64_t K, void* workspace, size_t workspace_bytes,
                                        void* stream) {
    if (int rc = dgrad_check_block(dy, wq, absmax, dx, 4, block, M, N, K)) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (act_dtype == QUANTA_BF16) {
        using T = __nv_bfloat16;
        return dgrad_launch<T, 4>((const T*)dy, wq, absmax, absmax, block, (T*)dx, M, N, K, workspace, workspace_bytes, st, 1);
    }
    if (act_dtype == QUANTA_F16) {
        using T = __half;
        return dgrad_launch<T, 4>((const T*)dy, wq, absmax, absmax, block, (T*)dx, M, N, K, workspace, workspace_bytes, st, 1);
    }
    return QUANTA_EINVAL;
}

extern "C" int quanta_int8_outlier_dgrad(const void* dy, int act_dtype, const int8_t* qw, const float* cw, void* dx, int64_t M,
                                         int64_t N, int64_t K, void* workspace, size_t workspace_bytes, void* stream) {
    if (int rc = dgrad_check(dy, qw, cw, dx, true, M, N, K)) return rc;
    if (K % 16 != 0) return QUANTA_EUNSUPPORTED;                                     // TMA row pitch of qw and dx
    const uint8_t* w = reinterpret_cast<const uint8_t*>(qw);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (act_dtype == QUANTA_BF16) {
        using T = __nv_bfloat16;
        return dgrad_launch<T, 8, true>((const T*)dy, w, cw, nullptr, 0, (T*)dx, M, N, K, workspace, workspace_bytes, st, 0);
    }
    if (act_dtype == QUANTA_F16) {
        using T = __half;
        return dgrad_launch<T, 8, true>((const T*)dy, w, cw, nullptr, 0, (T*)dx, M, N, K, workspace, workspace_bytes, st, 0);
    }
    return QUANTA_EINVAL;
}
