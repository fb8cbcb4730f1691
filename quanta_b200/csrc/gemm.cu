// W4A16 / W8A16 dequantize-then-matmul on the 5th-generation tensor cores
// (rows G1/G2 of SURVEY §8): y[M,N] = x[M,K] . dequant(Wq)[N,K]^T + bias.
//
// Mapping ("swap-AB"): the 128 output features of a weight tile are the UMMA M
// dimension (one TMEM lane each), the batch rows are the UMMA N dimension
// (16..256), so small batches do not waste the 128-row MMA:
//     D[n, m] (fp32, TMEM) += A[n, k] (dequantized weights, TMEM) * B[m, k] (x, smem)
// The dequantized A operand never touches shared memory: the dequant warps write
// it straight into tensor memory (tcgen05.st) and the MMA reads A from TMEM.
//
// Persistent, warp-specialised CTA (one per SM), 24 warps:
//   warp 0      TMA ring of raw weight codes: stages of [128 rows x 128 B] (SWIZZLE_128B),
//               i.e. 256 K values of 4-bit or 128 of 8-bit codes per box
//   warp 1      TMA ring of activation tiles [mb x 64] (SWIZZLE_128B, K-major B operand)
//   warp 2      TMEM allocation; one lane issues tcgen05.mma.kind::f16 (4 x K=16 per 64-K block)
//   warps 4-7   epilogue: tcgen05.ld the accumulator, add bias, store y — or store an fp32
//               partial and let the last-arriving CTA of the tile reduce all partials
//   warps 8-23  dequantize: 2 groups x 8 warps; a group owns every other stage and its own half of
//               the A slots and raw slots (so every mbarrier has one producer and one consumer
//               side and parity waits are unambiguous); a thread owns half a 64-K block of one
//               weight row (= its TMEM lane): 32 codes -> 16-bit A values -> one tcgen05.st
// Work is split stream-K style: the (tile, K-stage) units are cut into G equal
// contiguous ranges, one per CTA, so all SMs stream weights for the same time.
#include "gemm_tc.cuh"

namespace quanta {

constexpr int kASlots = 8;           // dequantized A tiles resident in TMEM
constexpr int kACols = kBlockK / 2;  // 32-bit TMEM columns per A slot (two 16-bit values per column)
constexpr int kDBase = kASlots * kACols;   // accumulators start at TMEM column 256
constexpr int kCtrlWarps = 4, kEpiWarps = 4, kDqGroups = 2, kDqGroupWarps = 8, kDqWarps = kDqGroupWarps * kDqGroups;
constexpr int kFirstEpiWarp = kCtrlWarps, kFirstDqWarp = kCtrlWarps + kEpiWarps;
constexpr int kGemmThreads = 32 * (kCtrlWarps + kEpiWarps + kDqWarps);

template <typename ACT, int BITS, int NOUT>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_wna16_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_x,
                  const __grid_constant__ CUtensorMap tmap_s, const __grid_constant__ CUtensorMap tmap_z,
                  const __grid_constant__ GemmOutputs<NOUT> outs, const float* __restrict__ scale, const float* __restrict__ zp, const ACT* __restrict__ bias,
                  unsigned int* __restrict__ counters, float* __restrict__ partial,
                  const __grid_constant__ GemmParams p) {
    using AT = ActTraits<ACT>;
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t raw_full[kMaxRing], raw_empty[kMaxRing], x_full[kMaxRing], x_empty[kMaxRing];
    __shared__ uint64_t a_full[kDqGroups], a_empty[kDqGroups], d_full[2], d_empty[2];
    __shared__ uint32_t tmem_base_slot;
    __shared__ int fix_flag;
    __shared__ int fin_tile;            // tile whose stream-K fix-up is done by the whole CTA at the end (-1: none)
    __shared__ __align__(1024) float stage[16][kTileN];        // epilogue transpose buffer (8 KB)
    __shared__ uint32_t nf4_pairs[256];                        // NF4: byte -> (level[lo nibble], level[hi nibble]) in the act type

    const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);       // warp-uniform for the compiler
    const unsigned int cta = blockIdx.x;

    // shared memory: [raw ring: raw_stages x 16|32 KB][x ring: x_stages x (xkb x mb x 128 B)]
    auto r_addr = [&](int s) { return smem + (uint32_t)s * p.raw_bytes; };
    auto x_addr = [&](int s) { return smem + p.x_ring_off + (uint32_t)s * p.x_slot_bytes; };

    SegWalk walk;
    walk.init(p, cta);
    int tile, s0, s1;
    if (tid == 32 * kFirstEpiWarp) fin_tile = -1;       // before the CTA-wide barrier below
    if (BITS == 4 && p.nf4 && tid >= 32 * kFirstDqWarp && tid < 32 * kFirstDqWarp + 256) {
        const int b = tid - 32 * kFirstDqWarp;      // visible to the dequant warps after the CTA-wide barrier below
        nf4_pairs[b] = AT::pack(kNf4Levels[b & 15], kNf4Levels[b >> 4]);
    }

    // Programmatic dependent launch: the next kernel on the stream may start its prologue while this grid is in
    // its tail; symmetrically this grid may have started during the previous kernel's tail, so everything that
    // depends on that kernel — the activation loads, bias, every global write — sits behind griddepcontrol.wait.
    // The weight stream (codes, scales, zero-points) does not and starts at once.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // Each producer initialises its own ring, checks in at the CTA-wide barrier without waiting
    // (barrier.arrive) and starts streaming at once; everybody else sees all barriers after
    // barrier.sync.  Producer loops are warp-uniform with one elected lane issuing, so the TMA
    // operands stay in uniform registers.
    if (warp == 0) {
        // ===== raw weight codes: deep TMA ring (bytes in flight hide the HBM latency) =====
        constexpr uint32_t kRawCodeBytes = BITS == 4 ? 16384u : 32768u;
        if (lane == 0) {
            for (int s = 0; s < p.raw_stages; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], kDqGroupWarps); }
            fence_barrier_init();
            prefetch_tensormap(&tmap_w);
            if (p.vec4) { prefetch_tensormap(&tmap_s); prefetch_tensormap(&tmap_z); }
        }
        __syncwarp();
        asm volatile("barrier.arrive 2, %0;" ::"n"(kGemmThreads) : "memory");
        const uint64_t pol_w = policy_evict_first();         // weights are streamed once
        int slot = 0, issued = 0;
        uint32_t ph = 0;
        while (walk.next(tile, s0, s1)) {
            int n_idx, m_idx;
            split_tile(tile, p, n_idx, m_idx);
            const int n0 = n_idx * kTileN;
            for (int s = s0; s < s1; ++s) {
                if (issued >= p.raw_stages) mbar_wait(&raw_empty[slot], ph ^ 1);
                if (elect_one()) {
                    mbar_arrive_expect_tx(&raw_full[slot], p.raw_bytes);
                    const uint32_t bar = smem_u32(&raw_full[slot]);
                    if (BITS == 4) {
                        tma_load_2d_plain(r_addr(slot), &tmap_w, bar, s * 128, n0, pol_w);
                    } else {
                        tma_load_2d_plain(r_addr(slot), &tmap_w, bar, s * 256, n0, pol_w);
                        tma_load_2d_plain(r_addr(slot) + 16384u, &tmap_w, bar, s * 256 + 128, n0, pol_w);
                    }
                    if (p.vec4) {
                        // the stage's scales and zero-points ride on the same barrier: [128 rows x 4 floats] each
                        tma_load_2d_plain(r_addr(slot) + kRawCodeBytes, &tmap_s, bar, s * kKbPerStage, n0, pol_w);
                        tma_load_2d_plain(r_addr(slot) + kRawCodeBytes + 2048u, &tmap_z, bar, s * kKbPerStage, n0, pol_w);
                    }
                }
                __syncwarp();
                ++issued;
                if (++slot == p.raw_stages) { slot = 0; ph ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===== activation tiles: xkb 64-K blocks per slot =====
        if (lane == 0) {
            for (int s = 0; s < p.x_stages; ++s) { mbar_init(&x_full[s], 1); mbar_init(&x_empty[s], 1); }
            fence_barrier_init();
            prefetch_tensormap(&tmap_x);
        }
        __syncwarp();
        asm volatile("barrier.arrive 2, %0;" ::"n"(kGemmThreads) : "memory");
        const uint64_t pol_x = policy_evict_last();          // activations are re-read by every CTA
        asm volatile("griddepcontrol.wait;" ::: "memory");   // x may be the previous kernel's output
        int slot = 0, issued = 0;
        uint32_t ph = 0;
        while (walk.next(tile, s0, s1)) {
            int n_idx, m_idx;
            split_tile(tile, p, n_idx, m_idx);
            const int m0 = m_idx * p.mb;
            for (int s = s0; s < s1; ++s) {
                for (int j = 0; j < kKbPerStage; j += p.xkb) {
                    if (issued >= p.x_stages) mbar_wait(&x_empty[slot], ph ^ 1);
                    if (elect_one()) {
                        mbar_arrive_expect_tx(&x_full[slot], p.x_slot_bytes);
                        // blocks past the end of K are out of bounds and arrive zero-filled
                        for (int jj = 0; jj < p.xkb; ++jj)
                            tma_load_2d_plain(x_addr(slot) + (uint32_t)jj * p.x_kb_bytes, &tmap_x, smem_u32(&x_full[slot]),
                                              (s * kKbPerStage + j + jj) * kBlockK, m0, pol_x);
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
            for (int s = 0; s < kDqGroups; ++s) { mbar_init(&a_full[s], kDqGroupWarps); mbar_init(&a_empty[s], 1); }
            for (int s = 0; s < 2; ++s) { mbar_init(&d_full[s], 1); mbar_init(&d_empty[s], kEpiWarps); }
            fence_barrier_init();
        }
        __syncwarp();
        tc_fence_before();
        asm volatile("barrier.sync 2, %0;" ::"n"(kGemmThreads) : "memory");
    }
    tc_fence_after();
    const uint32_t tmem = tmem_base_slot;

    if (warp == 2) {
        // ===== MMA issuer: the whole warp walks the schedule, one elected lane issues =====
        // (one issuer is enough: the body is bound by the dequant groups, not by the ~70 cycles of
        // dispatch per tcgen05.mma; DESIGN §4.1)
        const uint32_t idesc = (1u << 4) | (AT::kFmt << 7) | (AT::kFmt << 10) |
                               ((uint32_t)(p.mb >> 3) << 17) | ((uint32_t)(kTileN >> 4) << 24);
        const uint32_t kb_desc = p.x_kb_bytes >> 4;          // descriptor step between 64-K blocks of one slot
        const uint32_t nacc = (uint32_t)p.nacc;
        int sx = 0, seg = 0, sc = 0;
        uint32_t px = 0;
        while (walk.next(tile, s0, s1)) {
            const int buf = p.nbuf == 2 ? (seg & 1) : 0;
            const uint32_t use = (uint32_t)(p.nbuf == 2 ? (seg >> 1) : seg);      // how often `buf` was used before
            mbar_wait(&d_empty[buf], (use & 1) ^ 1);   // the epilogues have drained this accumulator
            const uint32_t tmem_d = tmem + kDBase + (uint32_t)(buf * p.nacc * p.mb);
            uint32_t touched = 0;                            // accumulators already written in this segment
            for (int s = s0; s < s1; ++s, ++sc) {
                const int nkb = min(kKbPerStage, p.total_kb - s * kKbPerStage);
                const int g = sc & 1;                        // dequant group = A buffer
                mbar_wait(&a_full[g], (uint32_t)(sc >> 1) & 1u);   // the stage's 4 A tiles are in TMEM
                const uint32_t ta = tmem + (uint32_t)(g * kKbPerStage * kACols);
#pragma unroll
                for (int j = 0; j < kKbPerStage; ++j) {
                    const int jj = j & (p.xkb - 1);
                    if (jj == 0) mbar_wait(&x_full[sx], px);       // activation slot landed
                    tc_fence_after();
                    const bool live = j < nkb;
                    uint32_t acc_idx[4], acc_flag[4];    // computed by every lane: stays warp-uniform
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        acc_idx[k] = (uint32_t)(4 * j + k) & (nacc - 1u);
                        acc_flag[k] = (touched >> acc_idx[k]) & 1u;
                        if (live) touched |= 1u << acc_idx[k];
                    }
                    if (elect_one()) {
                        if (live) {
                            const uint64_t db = smem_desc_sw128(x_addr(sx)) + (uint64_t)(jj * kb_desc);
#pragma unroll
                            for (int k = 0; k < kBlockK / 16; ++k)    // K = 16 per MMA: 8 TMEM columns of A, 32 bytes of B
                                umma_f16_ts(tmem_d + acc_idx[k] * (uint32_t)p.mb, ta + (uint32_t)(j * kACols + 8 * k),
                                            db + 2 * k, idesc, acc_flag[k]);
                        }
                        // both arrive when the MMAs above have read their operands
                        if (jj == p.xkb - 1) umma_commit(&x_empty[sx]);
                        if (j == kKbPerStage - 1) umma_commit(&a_empty[g]);
                    }
                    __syncwarp();
                    if (jj == p.xkb - 1) { if (++sx == p.x_stages) { sx = 0; px ^= 1; } }
                }
            }
            if (elect_one()) umma_commit(&d_full[buf]);
            __syncwarp();
            ++seg;
        }
    } else if (warp >= kFirstEpiWarp && warp < kFirstDqWarp) {
        // ===== epilogue: TMEM lane = output feature =====
        asm volatile("griddepcontrol.wait;" ::: "memory");   // bias reads, y / partial / counter writes
        const int quarter = warp & 3;
        const int row = 32 * quarter + lane;
        const int etid = tid - 32 * kFirstEpiWarp;
        if (etid == 0 && p.y_tma) { for (int o = 0; o < (NOUT == 1 ? 1 : p.n_out); ++o) prefetch_tensormap(&outs.maps[o]); }
        int seg = 0;
        while (walk.next(tile, s0, s1)) {
            const int buf = p.nbuf == 2 ? (seg & 1) : 0;
            const uint32_t use = (uint32_t)(p.nbuf == 2 ? (seg >> 1) : seg);
            int n_tile, m_tile;
            split_tile(tile, p, n_tile, m_tile);
            const int gn = n_tile * kTileN + row, m0 = m_tile * p.mb;
            const bool n_ok = gn < p.N;
            const int m_valid = min(p.mb, p.M - m0);
            const bool whole = (s0 == 0 && s1 == p.S);
            const bool last_seg = walk.u >= walk.u1;                  // no further segment for this CTA
            const float b = (bias != nullptr && n_ok) ? AT::to_float(bias[gn]) : 0.0f;
            // this CTA's partial slot for the tile: 0 if the tile is the first one the CTA touches, else 1
            const int which = (tile == tile_of_unit(first_unit(cta, p), p)) ? 0 : 1;
            float* mine = partial + ((size_t)cta * 2 + which) * (size_t)(kTileN * p.mb);

            mbar_wait(&d_full[buf], use & 1);
            tc_fence_after();
            const uint32_t taddr = tmem + ((uint32_t)(32 * quarter) << 16) + kDBase + (uint32_t)(buf * p.nacc * p.mb);
            // store mapping: thread -> 4 consecutive features (f4..f4+3), batch rows etid/32 + 4q
            const int f4 = 4 * (etid & 31);
            const int gn4 = n_tile * kTileN + f4;
            float b4[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) b4[e] = (bias != nullptr && gn4 + e < p.N) ? AT::to_float(bias[gn4 + e]) : 0.0f;
            const bool vec_ok = p.vec_store && gn4 + 3 < p.N;
            // accumulators the MMA warp wrote in this segment: 4 MMAs per 64-K block, rotating over nacc
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
                    // Whole tile: bias, 16-bit conversion, [16 rows x 128 features] staged in shared memory
                    // (two 4 KB buffers), then ONE TMA store per chunk; rows past M / features past N are
                    // clipped by the tensor map.  (Plain global stores from this kernel cost ~10 cycles
                    // per warp-store per SM: 20K cycles for a 128 x 256 tile.)
                    ACT* sbuf = reinterpret_cast<ACT*>(&stage[0][0]) + ((c0 >> 4) & 1) * (16 * kTileN);
                    if (etid == 0 && c0 >= 32) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // buffer's previous store has read it
                    asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
#pragma unroll
                    for (int j = 0; j < 16; ++j) sbuf[j * kTileN + row] = AT::from_float(__uint_as_float(r[j]) + b);
                    fence_proxy_async_smem();
                    asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
                    if (etid == 0 && c0 < m_valid) {
                        // one store per output buffer: the local y, or every tensor-parallel peer's y over NVLink
                        for (int o = 0; o < (NOUT == 1 ? 1 : p.n_out); ++o)
                            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                                         ::"l"(reinterpret_cast<uint64_t>(&outs.maps[o])), "r"(smem_u32(sbuf)),
                                           "r"(p.col0 + n_tile * kTileN), "r"(m0 + c0) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    continue;
                }
                // Otherwise transpose the chunk through shared memory so that the stores are full rows:
                // thread -> 4 consecutive features of 4 batch rows, 8 / 16 bytes per store.
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");      // previous chunk fully read
#pragma unroll
                for (int j = 0; j < 16; ++j) stage[j][row] = __uint_as_float(r[j]);
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
                if (c0 < m_valid) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int ml = 4 * q + (etid >> 5);              // batch row within the chunk
                        const int m = c0 + ml;
                        if (m < m_valid) {
                            const float4 v = *reinterpret_cast<const float4*>(&stage[ml][f4]);
                            if (whole) {
                                const float o[4] = {v.x + b4[0], v.y + b4[1], v.z + b4[2], v.w + b4[3]};
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
                            } else {
                                *reinterpret_cast<float4*>(mine + m * kTileN + f4) = v;
                            }
                        }
                    }
                }
            }
            if (whole && p.y_tma && etid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // staging free for the next segment
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&d_empty[buf]);   // accumulator may be overwritten
            if (!whole) {
                // stream-K fix-up: the CTA that arrives last at the tile's counter reduces every partial
                const unsigned int tu0 = (unsigned int)tile * (unsigned int)p.S;
                const int c_first = cta_of_unit(tu0, p), c_last = cta_of_unit(tu0 + (unsigned int)p.S - 1u, p);
                // release: CTA barrier, then one thread publishes with a gpu-scope fence + atomic (fences
                // are cumulative over the barrier); acquire on the way back mirrors it
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
                if (etid == 0) {
                    __threadfence();
                    const unsigned int old = atomicAdd(&counters[tile], 1u);
                    __threadfence();
                    const int last = (old == (unsigned int)(c_last - c_first)) ? 1 : 0;
                    if (last) counters[tile] = 0u;      // leave the workspace clean for the next call
                    fix_flag = last;
                }
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
                if (fix_flag) {
                    if (last_seg && p.mb >= 64) {
                        // the CTA has nothing left to do: hand the reduction to all 20 epilogue + dequant
                        // warps (5x the loads in flight) after the role loops
                        if (etid == 0) fin_tile = tile;
                    } else {
                        fixup_reduce<ACT, NOUT>(p, outs, bias, partial, tile, etid, 32 * kEpiWarps);
                    }
                }
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");      // fix_flag is reused
            }
            ++seg;
        }
    } else if (warp >= kFirstDqWarp) {
        // ===== dequantize: thread = (weight row = TMEM lane, half of each 64-K block) =====
        using V2 = typename AT::V2;
        const int quarter = warp & 3;                                  // TMEM lane quarter this warp may access
        const int half = ((warp - kFirstDqWarp) >> 2) & 1;            // which 32 of the 64 K values
        const int group = (warp - kFirstDqWarp) / kDqGroupWarps;      // stages group, group + 2, ...
        const int row = 32 * quarter + lane;
        // this group's A buffer: 4 tiles of 32 columns; this thread's half tile starts 16 columns in
        const uint32_t a_addr = tmem + ((uint32_t)(32 * quarter) << 16) + (uint32_t)(group * kKbPerStage * kACols + 16 * half);
        const V2 c2 = AT::dup(AT::kCentre);
        // Scale / zero-point of a stage: delivered by TMA next to the raw codes (vec4), else loaded
        // with plain loads one stage of work ahead (odd shapes: K not a multiple of 256, block > 64).
        constexpr uint32_t kRawCodeBytes = BITS == 4 ? 16384u : 32768u;
        SegWalk ahead = walk;
        int a_tile = 0, a_s = 0, a_s1 = 0;
        bool a_ok = ahead.next(a_tile, a_s, a_s1);
        float sv[4], zv[4];
        auto fetch_params = [&](int t, int s) {
            int n_idx, m_idx;
            split_tile(t, p, n_idx, m_idx);
            const int gn = n_idx * kTileN + row;
            const int64_t rbase = (int64_t)(gn < p.N ? gn : p.N - 1) * p.scale_stride;
            const int kb = s * kKbPerStage;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int col = min(kb + j, p.total_kb - 1) >> p.block_shift;
                sv[j] = __ldg(scale + rbase + col);
                zv[j] = __ldg(zp + rbase + col);
            }
        };
        // advance `ahead` by n stages (across segments)
        auto skip = [&](int n) {
            while (a_ok && n > 0) {
                const int room = a_s1 - a_s;
                if (n < room) { a_s += n; n = 0; }
                else { n -= room; a_ok = ahead.next(a_tile, a_s, a_s1); }
            }
        };
        if (!p.vec4) {
            skip(group);
            if (a_ok) fetch_params(a_tile, a_s);
        }

        int sc = 0;                 // global stage counter of this CTA
        int rslot = 0;
        uint32_t rph = 0;
        while (walk.next(tile, s0, s1)) {
            for (int s = s0; s < s1; ++s, ++sc) {
                if ((sc & (kDqGroups - 1)) == group) {
                    const int nkb = min(kKbPerStage, p.total_kb - s * kKbPerStage);
                    float cs[4], cz[4];
                    if (!p.vec4) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) { cs[j] = sv[j]; cz[j] = zv[j]; }
                        skip(kDqGroups);
                        if (a_ok) fetch_params(a_tile, a_s); // lands while this stage is processed
                    }
                    mbar_wait(&raw_full[rslot], rph);

                    const uint32_t rrow = r_addr(rslot) + (uint32_t)row * 128u;
                    const uint32_t sw = (uint32_t)(row & 7);
                    if (p.vec4) {
                        const uint4 a = lds128g(r_addr(rslot) + kRawCodeBytes + (uint32_t)row * 16u);
                        const uint4 c = lds128g(r_addr(rslot) + kRawCodeBytes + 2048u + (uint32_t)row * 16u);
                        cs[0] = __uint_as_float(a.x); cs[1] = __uint_as_float(a.y); cs[2] = __uint_as_float(a.z); cs[3] = __uint_as_float(a.w);
                        cz[0] = __uint_as_float(c.x); cz[1] = __uint_as_float(c.y); cz[2] = __uint_as_float(c.z); cz[3] = __uint_as_float(c.w);
                    }
                    // the MMAs that read this group's A buffer two stages ago are done
                    mbar_wait(&a_empty[group], ((uint32_t)(sc >> 1) & 1u) ^ 1u);
                    tc_fence_after();
#pragma unroll
                    for (int j = 0; j < kKbPerStage; ++j) {
                        if (j < nkb) {
                            uint32_t out[16];
                            if (BITS == 4 && p.nf4) {
                                // NF4: one shared-memory lookup per code byte gives the K-adjacent pair
                                // (level[lo], level[hi]); one packed multiply applies the block's abs_max
                                const V2 s2 = AT::dup(cs[j]);
                                const uint4 rv = lds128g(rrow + (((uint32_t)(2 * j + half) ^ sw) << 4));
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
                            } else if (BITS == 4) {
                                const V2 s2 = AT::dup(cs[j]);
                                const V2 z2 = AT::dup(__fmaf_rn(8.0f, cs[j], cz[j]));
                                const uint4 rv = lds128g(rrow + (((uint32_t)(2 * j + half) ^ sw) << 4));
                                dequant_word4<ACT>(rv.x, s2, z2, c2, out);
                                dequant_word4<ACT>(rv.y, s2, z2, c2, out + 4);
                                dequant_word4<ACT>(rv.z, s2, z2, c2, out + 8);
                                dequant_word4<ACT>(rv.w, s2, z2, c2, out + 12);
                            } else {
                                const float zc = __fmaf_rn(-32768.0f, cs[j], cz[j]);
                                const uint32_t box = rrow + (uint32_t)(j >> 1) * 16384u;
#pragma unroll
                                for (int h = 0; h < 2; ++h) {
                                    const uint4 rv = lds128g(box + (((uint32_t)(4 * (j & 1) + 2 * half + h) ^ sw) << 4));
                                    dequant_word8<ACT>(rv.x, cs[j], zc, out + 8 * h);
                                    dequant_word8<ACT>(rv.y, cs[j], zc, out + 8 * h + 2);
                                    dequant_word8<ACT>(rv.z, cs[j], zc, out + 8 * h + 4);
                                    dequant_word8<ACT>(rv.w, cs[j], zc, out + 8 * h + 6);
                                }
                            }
                            tmem_st16(a_addr + (uint32_t)(j * kACols), out);
                        }
                        }
                    tmem_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        mbar_arrive(&a_full[group]);
                        mbar_arrive(&raw_empty[rslot]);
                    }

                }
                if (++rslot == p.raw_stages) { rslot = 0; rph ^= 1; }
            }
        }
    }

    if (warp >= kFirstEpiWarp && p.mb >= 64) {
        // epilogue + dequant warps: a pending last-segment fix-up is reduced by all of them (small
        // batches have too few rows to share: the epilogue warps did it in their loop)
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("bar.sync 3, %0;" ::"n"(32 * (kEpiWarps + kDqWarps)) : "memory");
        const int ft = *reinterpret_cast<volatile int*>(&fin_tile);
        if (ft >= 0)
            fixup_reduce<ACT, NOUT>(p, outs, bias, partial, ft, tid - 32 * kFirstEpiWarp, 32 * (kEpiWarps + kDqWarps));
    }
    if (tid == 32 * kFirstEpiWarp) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");       // y stores have landed
    tc_fence_before();
    __syncthreads();
    if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem, kTmemCols); }
}

// ---- host side --------------------------------------------------------------

size_t gemm_workspace_bytes(int64_t M, int64_t) {
    int64_t mb = (M + 31) / 32 * 32;
    if (mb > 256) mb = 256;
    return (size_t)kCounterBytes + (size_t)kNumSMs * 2 * kTileN * (size_t)mb * sizeof(float) + 512;
}

template <typename ACT, int BITS, int NOUT>
static int gemm_tc_launch(GemmParams& p, const ACT* x, const uint8_t* wq, const float* scale, const float* zp,
                          const ACT* bias, void* const* ys, int64_t M, int64_t N, int64_t K, void* workspace, size_t ws_bytes,
                          cudaStream_t st) {
    const int mb = p.mb;
    const int tiles = p.n_tiles * p.m_tiles;
    if (tiles > kMaxTiles) return QUANTA_EUNSUPPORTED;
    if ((unsigned long long)tiles * (unsigned long long)p.S * (unsigned long long)(kNumSMs + 1) >= (1ull << 32)) return QUANTA_EUNSUPPORTED;
    p.U = (unsigned int)tiles * (unsigned int)p.S;
    p.G = choose_units(tiles, p.S, mb, BITS == 4 ? 16384 : 32768);
    p.uq = p.U / (unsigned int)p.G;
    p.ur = p.U % (unsigned int)p.G;
    {
        // x / d == __umulhi(x, ceil(2^32 / d)) for every x <= xmax when xmax * (magic * d - 2^32) < 2^32
        auto magic_for = [](unsigned int d, unsigned long long xmax, unsigned int* out) {
            if (d == 1) { *out = 0u; return true; }
            const unsigned long long m = ((1ull << 32) + d - 1ull) / d;
            *out = (unsigned int)m;
            return xmax * (m * d - (1ull << 32)) < (1ull << 32);
        };
        if (!magic_for((unsigned int)p.S, p.U, &p.s_magic) || !magic_for((unsigned int)p.n_tiles, (unsigned long long)tiles, &p.nt_magic))
            return QUANTA_EUNSUPPORTED;
    }
    p.x_kb_bytes = (uint32_t)mb * 128u;                     // one 64-K block of the activation tile
    p.xkb = p.x_kb_bytes <= 8192u ? 4 : (p.x_kb_bytes <= 16384u ? 2 : 1);    // activation slots of at most 32 KB
    p.x_slot_bytes = p.x_kb_bytes * (uint32_t)p.xkb;
    p.raw_bytes = (BITS == 4 ? 16384u : 32768u) + (p.vec4 ? 4096u : 0u);    // codes (+ scale / zero-point tiles)
    // Shared-memory budget: an activation ring sized for the MMA, everything else for the raw-code
    // ring — raw bytes in flight are what hides the HBM latency.
    const uint32_t budget = 214u * 1024u;
    int x_stages = p.x_slot_bytes <= 8192u ? 6 : (p.x_slot_bytes <= 16384u ? 4 : (p.x_kb_bytes <= 8192u ? 3 : 4));
    int raw_stages = (int)((budget - (uint32_t)x_stages * p.x_slot_bytes) / p.raw_bytes);
    if (raw_stages > kMaxRing) raw_stages = kMaxRing;
    raw_stages &= ~1;                  // even: a raw slot is always consumed by the same dequant group
    if (raw_stages < 2) return QUANTA_EUNSUPPORTED;
    p.raw_stages = raw_stages;
    p.x_stages = x_stages;
    p.x_ring_off = (uint32_t)raw_stages * p.raw_bytes;

    const size_t need = (size_t)kCounterBytes + (size_t)p.G * 2 * kTileN * (size_t)mb * sizeof(float) + 256;
    if (!workspace || ws_bytes < need) return QUANTA_EWORKSPACE;
    uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    unsigned int* counters = reinterpret_cast<unsigned int*>(ws);
    float* partial = reinterpret_cast<float*>(ws + kCounterBytes);

    CUtensorMap tmap_w, tmap_x;
    const uint64_t wrow_bytes = (uint64_t)K * BITS / 8;
    int rc = make_tensor_map_2d(&tmap_w, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, wq, wrow_bytes, (uint64_t)N, wrow_bytes,
                                128, kTileN, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = make_tensor_map_2d(&tmap_x, ActTraits<ACT>::kTma, 2, x, (uint64_t)K, (uint64_t)M, (uint64_t)K * 2, kBlockK,
                            (uint32_t)mb, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;

    CUtensorMap tmap_s = tmap_w, tmap_z = tmap_w;          // placeholders unless the parameters ride on TMA
    if (p.vec4) {
        rc = make_tensor_map_2d(&tmap_s, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, scale, (uint64_t)p.scale_stride, (uint64_t)N,
                                (uint64_t)p.scale_stride * 4, kKbPerStage, kTileN, CU_TENSOR_MAP_SWIZZLE_NONE);
        if (rc) return rc;
        rc = make_tensor_map_2d(&tmap_z, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, zp, (uint64_t)p.scale_stride, (uint64_t)N,
                                (uint64_t)p.scale_stride * 4, kKbPerStage, kTileN, CU_TENSOR_MAP_SWIZZLE_NONE);
        if (rc) return rc;
    }
    GemmOutputs<NOUT> outs;
    bool aligned16 = true, aligned8 = true;
    for (int o = 0; o < NOUT; ++o) {
        outs.maps[o] = tmap_w;                              // placeholder
        outs.y[o] = o < p.n_out ? ys[o] : nullptr;
        if (o < p.n_out) {
            aligned16 = aligned16 && (reinterpret_cast<uintptr_t>(ys[o]) & 15) == 0;
            aligned8 = aligned8 && (reinterpret_cast<uintptr_t>(ys[o]) & 7) == 0;
        }
    }
    p.vec_store = (aligned8 && (p.ldy & 3) == 0 && (p.col0 & 3) == 0) ? 1 : 0;
    p.y_tma = (aligned16 && (p.ldy & 7) == 0) ? 1 : 0;
    if (p.y_tma) {
        // window [M, col0 + N] of each buffer: features past this call's columns are clipped by the map
        for (int o = 0; o < p.n_out; ++o) {
            rc = make_tensor_map_2d(&outs.maps[o], ActTraits<ACT>::kTma, 2, ys[o], (uint64_t)(p.col0 + N), (uint64_t)M,
                                    (uint64_t)p.ldy * 2, kTileN, 16, CU_TENSOR_MAP_SWIZZLE_NONE);
            if (rc) return rc;
        }
    }
    auto kern = gemm_wna16_kernel<ACT, BITS, NOUT>;
    const int smem = (int)(p.x_ring_off + (uint32_t)p.x_stages * p.x_slot_bytes + 1024);
    if (int e = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), smem)) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)p.G);
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tmap_w, tmap_x, tmap_s, tmap_z, outs, scale, zp, bias, counters, partial, p);
    return cuda_status(e != cudaSuccess ? e : cudaGetLastError());
}

// mma.sync weight-stream kernel for decode-sized batches (gemm_small.cu)
bool gemm_small_eligible(int64_t M, int64_t N, int64_t K, int64_t block, const void* scale, const void* zp);
template <typename ACT, int BITS>
int gemm_small_launch(const ACT* x, const uint8_t* wq, const float* scale, const float* zp, const ACT* bias, void* const* ys,
                      int n_out, int64_t ldy, int64_t col0, int64_t M, int64_t N, int64_t K, void* workspace, size_t ws_bytes,
                      cudaStream_t st, int nf4, const PeerSync* sync);

template <typename ACT, int BITS>
static int gemm_launch(const ACT* x, const uint8_t* wq, const float* scale, const float* zp, int64_t block,
                       const ACT* bias, ACT* y, int64_t M, int64_t N, int64_t K, void* workspace, size_t ws_bytes,
                       cudaStream_t st, int nf4 = 0, void* const* ys = nullptr, int n_out = 1, int64_t ldy = 0,
                       int64_t col0 = 0, const PeerSync* sync = nullptr) {
    void* one[1] = {y};
    if (!ys) { ys = one; n_out = 1; ldy = N; col0 = 0; }
    // M <= 16: the weight-stream kernel (HBM-bound regime; gemm_small.cu)
    if (gemm_small_eligible(M, N, K, block, scale, zp))
        return gemm_small_launch<ACT, BITS>(x, wq, scale, zp, bias, ys, n_out, ldy, col0, M, N, K, workspace, ws_bytes, st, nf4, sync);
    if (sync) return QUANTA_EUNSUPPORTED;                    // the in-kernel completion exists in the small-batch kernel only
    GemmParams p;
    p.M = (int)M; p.N = (int)N; p.K = (int)K;
    int mb = (int)((M + 15) / 16 * 16);
    if (mb > 256) mb = 256;
    p.mb = mb;
    p.m_tiles = (int)((M + mb - 1) / mb);
    p.n_tiles = (int)((N + kTileN - 1) / kTileN);
    p.total_kb = (int)(K / kBlockK);
    p.S = (p.total_kb + kKbPerStage - 1) / kKbPerStage;
    // accumulators: nbuf x nacc x mb <= 256 TMEM columns
    p.nacc = mb <= 16 ? 8 : (mb <= 64 ? 4 : (mb <= 128 ? 2 : 1));
    p.nbuf = (2 * p.nacc * mb <= kTmemCols - kDBase) ? 2 : 1;
    p.nf4 = nf4;
    p.n_out = n_out; p.ldy = (int)ldy; p.col0 = (int)col0;
    p.scale_stride = (int)(K / block);
    int bs = 0; while ((int64_t)(kBlockK << bs) < block) ++bs;
    p.block_shift = bs;
    p.vec4 = (bs == 0 && (p.scale_stride & 3) == 0 &&
              ((reinterpret_cast<uintptr_t>(scale) | reinterpret_cast<uintptr_t>(zp)) & 15) == 0) ? 1 : 0;
    if (n_out > 1) return gemm_tc_launch<ACT, BITS, kMaxOut>(p, x, wq, scale, zp, bias, ys, M, N, K, workspace, ws_bytes, st);
    return gemm_tc_launch<ACT, BITS, 1>(p, x, wq, scale, zp, bias, ys, M, N, K, workspace, ws_bytes, st);
}

}  // namespace quanta

using namespace quanta;

extern "C" int quanta_gemm_wna16(const void* x, int act_dtype, const uint8_t* wq, int bits, const float* scale,
                                 const float* zp, int64_t block, const void* bias, void* y, int64_t M, int64_t N,
                                 int64_t K, void* workspace, size_t workspace_bytes, void* stream) {
    if (!x || !wq || !scale || !zp || !y || M <= 0 || N <= 0 || K <= 0) return QUANTA_EINVAL;
    if ((bits != 4 && bits != 8) || block <= 0 || block % kBlockK != 0 || K % block != 0) return QUANTA_EINVAL;
    if ((block / kBlockK) & (block / kBlockK - 1)) return QUANTA_EUNSUPPORTED;          // block = 64 * 2^j
    if ((K * bits / 8) % 16 != 0 || (K * 2) % 16 != 0) return QUANTA_EUNSUPPORTED;      // TMA row pitch
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(wq)) & 15) return QUANTA_EUNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (act_dtype == QUANTA_BF16) {
        using T = __nv_bfloat16;
        return bits == 4 ? gemm_launch<T, 4>((const T*)x, wq, scale, zp, block, (const T*)bias, (T*)y, M, N, K, workspace, workspace_bytes, st)
                         : gemm_launch<T, 8>((const T*)x, wq, scale, zp, block, (const T*)bias, (T*)y, M, N, K, workspace, workspace_bytes, st);
    }
    if (act_dtype == QUANTA_F16) {
        using T = __half;
        return bits == 4 ? gemm_launch<T, 4>((const T*)x, wq, scale, zp, block, (const T*)bias, (T*)y, M, N, K, workspace, workspace_bytes, st)
                         : gemm_launch<T, 8>((const T*)x, wq, scale, zp, block, (const T*)bias, (T*)y, M, N, K, workspace, workspace_bytes, st);
    }
    return QUANTA_EINVAL;
}

extern "C" int quanta_gemm_nf4a16(const void* x, int act_dtype, const uint8_t* wq, const float* absmax, int64_t block,
                                  const void* bias, void* y, int64_t M, int64_t N, int64_t K, void* workspace,
                                  size_t workspace_bytes, void* stream) {
    if (!x || !wq || !absmax || !y || M <= 0 || N <= 0 || K <= 0) return QUANTA_EINVAL;
    if (block <= 0 || block % kBlockK != 0 || K % block != 0) return QUANTA_EINVAL;
    if ((block / kBlockK) & (block / kBlockK - 1)) return QUANTA_EUNSUPPORTED;
    if ((K / 2) % 16 != 0 || (K * 2) % 16 != 0) return QUANTA_EUNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(wq)) & 15) return QUANTA_EUNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (act_dtype == QUANTA_BF16) {
        using T = __nv_bfloat16;
        return gemm_launch<T, 4>((const T*)x, wq, absmax, absmax, block, (const T*)bias, (T*)y, M, N, K, workspace, workspace_bytes, st, 1);
    }
    if (act_dtype == QUANTA_F16) {
        using T = __half;
        return gemm_launch<T, 4>((const T*)x, wq, absmax, absmax, block, (const T*)bias, (T*)y, M, N, K, workspace, workspace_bytes, st, 1);
    }
    return QUANTA_EINVAL;
}

static int gemm_scatter_entry(const void* x, int act_dtype, const uint8_t* wq, int bits, const float* scale,
                                         const float* zp, int64_t block, const void* bias, void* const* ys, int n_out,
                                         int64_t ldy, int64_t col0, int64_t M, int64_t N, int64_t K, void* workspace,
                                         size_t workspace_bytes, void* stream, const PeerSync* sync) {
    if (!x || !wq || !scale || !zp || !ys || n_out < 1 || n_out > kMaxOut || M <= 0 || N <= 0 || K <= 0) return QUANTA_EINVAL;
    if (ldy < col0 + N || col0 < 0) return QUANTA_EINVAL;
    for (int o = 0; o < n_out; ++o) if (!ys[o]) return QUANTA_EINVAL;
    if ((bits != 4 && bits != 8) || block <= 0 || block % kBlockK != 0 || K % block != 0) return QUANTA_EINVAL;
    if ((block / kBlockK) & (block / kBlockK - 1)) return QUANTA_EUNSUPPORTED;
    if ((K * bits / 8) % 16 != 0 || (K * 2) % 16 != 0) return QUANTA_EUNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(wq)) & 15) return QUANTA_EUNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (act_dtype == QUANTA_BF16) {
        using T = __nv_bfloat16;
        return bits == 4 ? gemm_launch<T, 4>((const T*)x, wq, scale, zp, block, (const T*)bias, nullptr, M, N, K, workspace, workspace_bytes, st, 0, ys, n_out, ldy, col0, sync)
                         : gemm_launch<T, 8>((const T*)x, wq, scale, zp, block, (const T*)bias, nullptr, M, N, K, workspace, workspace_bytes, st, 0, ys, n_out, ldy, col0, sync);
    }
    if (act_dtype == QUANTA_F16) {
        using T = __half;
        return bits == 4 ? gemm_launch<T, 4>((const T*)x, wq, scale, zp, block, (const T*)bias, nullptr, M, N, K, workspace, workspace_bytes, st, 0, ys, n_out, ldy, col0, sync)
                         : gemm_launch<T, 8>((const T*)x, wq, scale, zp, block, (const T*)bias, nullptr, M, N, K, workspace, workspace_bytes, st, 0, ys, n_out, ldy, col0, sync);
    }
    return QUANTA_EINVAL;
}

extern "C" int quanta_gemm_wna16_scatter(const void* x, int act_dtype, const uint8_t* wq, int bits, const float* scale,
                                         const float* zp, int64_t block, const void* bias, void* const* ys, int n_out,
                                         int64_t ldy, int64_t col0, int64_t M, int64_t N, int64_t K, void* workspace,
                                         size_t workspace_bytes, void* stream) {
    return gemm_scatter_entry(x, act_dtype, wq, bits, scale, zp, block, bias, ys, n_out, ldy, col0, M, N, K, workspace, workspace_bytes,
                              stream, nullptr);
}

// The same, with the ranks' synchronisation inside the kernel: when it has completed on this rank, every rank's columns
// have landed in this rank's buffer (see PeerSync in common.cuh) and no barrier kernel is needed behind it.
// QUANTA_EUNSUPPORTED when the shape is not served by the small-batch kernel (M > 16, block != 64, K % 256 != 0):
// the caller then uses quanta_gemm_wna16_scatter plus its own barrier.
extern "C" int quanta_gemm_wna16_scatter_sync(const void* x, int act_dtype, const uint8_t* wq, int bits, const float* scale,
                                              const float* zp, int64_t block, const void* bias, void* const* ys, int n_out,
                                              int64_t ldy, int64_t col0, int64_t M, int64_t N, int64_t K, void* workspace,
                                              size_t workspace_bytes, void* const* peer_flags, int rank, int world,
                                              unsigned int* epoch_counter, void* stream) {
    if (!peer_flags || !epoch_counter || world < 2 || world > 8 || rank < 0 || rank >= world) return QUANTA_EINVAL;
    PeerSync sync;
    for (int r = 0; r < 8; ++r) sync.flags[r] = r < world ? peer_flags[r] : nullptr;
    sync.rank = rank; sync.world = world; sync.epoch_counter = epoch_counter;
    return gemm_scatter_entry(x, act_dtype, wq, bits, scale, zp, block, bias, ys, n_out, ldy, col0, M, N, K, workspace, workspace_bytes,
                              stream, &sync);
}
