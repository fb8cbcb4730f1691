// Microbenchmark: the blockwise quantize stream (quantize_rows_tma_multi_kernel) without its arithmetic, under a
// STATIC persistent schedule: a grid of 2 CTAs per SM in which CTA b walks tiles b, b + grid, ...  The kernel claims
// tiles with cluster launch control instead and runs faster than this micro, so these numbers bound the static
// schedule, not the hardware.  Same geometry as the kernel: TMA boxes of 256 rows x 32 fp32 (SWIZZLE_128B) into a
// 3-stage ring, one producer lane, 256 consumer threads that each read their 128-byte row out of shared memory.  Over
// the bench step's working set (all 224 Llama-2-7B linears, 25.9 GB of fp32) it reports GB/s of reads for
//   read     : reads only (a row is consumed, nothing is written)
//   mix      : per row, 16 B of codes plus one scale and one zero point per 2 rows into two arrays, 0.625 B per
//              element read: the headline's write mix
//   mix P=k  : the mix with tile g + k * grid prefetched into L2 (cp.async.bulk.prefetch.tensor) before the producer
//              waits for the free stage of tile g, with and without an evict-first hint on the prefetch
// and, for each, the load's L2 policy evict-first and evict-normal (the kernel's).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o quantize_stream_ceiling quantize_stream_ceiling.cu
#include <cstdio>
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e_)); return 1; } } while (0)

constexpr int kRows = 256, kStages = 3, kThreads = kRows + 32, kTileBytes = kRows * 128;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t n) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(n)); }
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t ph) {
    asm volatile("{\n\t.reg .pred p;\n\tW_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra D_%=;\n\tbra W_%=;\n\tD_%=:\n\t}"
                 ::"r"(smem_u32(b)), "r"(ph) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory"); }
__device__ __forceinline__ void mbar_expect(uint64_t* b, uint32_t n) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(n) : "memory");
}

// MODE 0: read only; 1: the read/write mix.  pf: prefetch distance in tiles (0 = none); pf_hint: evict-first on the
// prefetch; load_first: evict-first on the load (else evict-normal).
template <int MODE>
__global__ void __launch_bounds__(kThreads, 2)
stream(const __grid_constant__ CUtensorMap map, int n_tiles, int pf, int pf_hint, int load_first, uint8_t* q, float* sc,
       float* zp) {
    extern __shared__ uint8_t raw[];
    __shared__ uint64_t full[kStages], empty[kStages];
    __shared__ int tile_of[kStages];
    __shared__ uint32_t scratch[kThreads / 32];
    const uint32_t smem = (smem_u32(raw) + 1023u) & ~1023u;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kRows / 32); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (warp == kRows / 32) {
        if (lane != 0) return;
        uint64_t pol, ppol;
        if (load_first) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
        else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(ppol));
        const int grid = gridDim.x;
        int g = blockIdx.x;
        for (int i = 0;; ++i, g += grid) {
            const int s = i % kStages;
            const uint32_t ph = (i / kStages) & 1;
            const int gp = g + pf * grid;
            if (pf > 0 && gp < n_tiles) {
                if (pf_hint)
                    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile.L2::cache_hint [%0, {%1, %2}], %3;"
                                 ::"l"((uint64_t)&map), "r"(0), "r"(gp * kRows), "l"(ppol) : "memory");
                else
                    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];"
                                 ::"l"((uint64_t)&map), "r"(0), "r"(gp * kRows) : "memory");
            }
            mbar_wait(&empty[s], ph ^ 1);
            if (g >= n_tiles) { tile_of[s] = -1; mbar_arrive(&full[s]); return; }
            tile_of[s] = g;
            mbar_expect(&full[s], kTileBytes);
            asm volatile(
                "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint"
                " [%0], [%1, {%3, %4}], [%2], %5;"
                ::"r"(smem + s * kTileBytes), "l"((uint64_t)&map), "r"(smem_u32(&full[s])), "r"(0), "r"(g * kRows), "l"(pol)
                : "memory");
        }
    }
    for (int i = 0;; ++i) {
        const int s = i % kStages;
        mbar_wait(&full[s], (i / kStages) & 1);
        const int t = *reinterpret_cast<volatile int*>(&tile_of[s]);
        if (t < 0) return;
        uint32_t x = 0;
        const uint32_t row = smem + s * kTileBytes + tid * 128;
        for (int j = 0; j < 8; ++j) {
            uint32_t a, b, c, d;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(row + ((j ^ (tid & 7)) << 4)));
            x ^= a ^ b ^ c ^ d;
        }
        __syncwarp();
        if (lane == 0) {       // the stage is free once every row of the warp has been read (see mbar_arrive_after_loads)
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(smem_u32(&scratch[warp])), "r"(x) : "memory");
            mbar_arrive(&empty[s]);
        }
        const int64_t r = (int64_t)t * kRows + tid;
        if (MODE == 0) {
            if (x == 0x7fc00001u) q[0] = 1;          // never true for the fill below; keeps the loads live
        } else {
            __stcs(reinterpret_cast<uint4*>(q + r * 16), make_uint4(x, x, x, x));
            if ((lane & 1) == 0) { sc[r >> 1] = __uint_as_float(x); zp[r >> 1] = __uint_as_float(x); }   // as the kernel: block b = row / 2
        }
    }
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int main() {
    // the bench step: 32 layers x (4 x 4096^2 + 3 x 11008 x 4096) fp32 elements
    const int64_t elems = 32LL * (4LL * 4096 * 4096 + 3LL * 11008 * 4096);
    const int64_t rows = elems / 32;
    const int n_tiles = (int)((rows + kRows - 1) / kRows);
    const double rd = (double)elems * 4, wr = (double)elems * 0.625;
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, 0));
    float *x = nullptr, *sc = nullptr, *zp = nullptr;
    uint8_t* q = nullptr;
    CK(cudaMalloc(&x, elems * 4));
    CK(cudaMalloc(&q, elems / 2));
    CK(cudaMalloc(&sc, rows / 2 * 4));
    CK(cudaMalloc(&zp, rows / 2 * 4));
    CK(cudaMemset(x, 0x3c, elems * 4));
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr));
    CUtensorMap map;
    cuuint64_t dims[2] = {32, (cuuint64_t)rows}, strides[1] = {128};
    cuuint32_t box[2] = {32, kRows}, es[2] = {1, 1};
    if (((EncodeFn)fn)(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, x, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE)) {
        printf("tensor map encode failed\n");
        return 1;
    }
    const int smem = kStages * kTileBytes + 1024;
    CK(cudaFuncSetAttribute(stream<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CK(cudaFuncSetAttribute(stream<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, stream<1>, kThreads, smem));
    const int grid = occ * p.multiProcessorCount;
    printf("{\"device\": \"%s\", \"sms\": %d, \"ctas_per_sm\": %d, \"grid\": %d, \"read_GB\": %.3f, \"mix_write_GB\": %.3f}\n",
           p.name, p.multiProcessorCount, occ, grid, rd / 1e9, wr / 1e9);
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    struct Cfg { int mode, pf, pf_hint, load_first; } cfgs[] = {
        {0, 0, 0, 1}, {0, 0, 0, 0}, {1, 0, 0, 1}, {1, 0, 0, 0},
        {1, 2, 0, 1}, {1, 2, 1, 1}, {1, 2, 0, 0}, {1, 4, 0, 1}, {1, 4, 1, 1}, {1, 4, 0, 0}};
    const int reps = 5;
    for (const Cfg& c : cfgs) {
        auto run = [&]() {
            if (c.mode == 0) stream<0><<<grid, kThreads, smem>>>(map, n_tiles, c.pf, c.pf_hint, c.load_first, q, sc, zp);
            else stream<1><<<grid, kThreads, smem>>>(map, n_tiles, c.pf, c.pf_hint, c.load_first, q, sc, zp);
        };
        run();
        CK(cudaDeviceSynchronize());
        float best = 1e30f, tot = 0;
        for (int r = 0; r < reps; ++r) {
            CK(cudaEventRecord(e0));
            run();
            CK(cudaEventRecord(e1));
            CK(cudaEventSynchronize(e1));
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, e0, e1));
            tot += ms;
            if (ms < best) best = ms;
        }
        CK(cudaGetLastError());
        const double bytes = rd + (c.mode ? wr : 0);
        printf("{\"case\": \"%s\", \"prefetch_tiles\": %d, \"prefetch_hint\": \"%s\", \"load_hint\": \"%s\", \"ms_best\": %.3f, "
               "\"ms_mean\": %.3f, \"read_GBps\": %.1f, \"total_GBps\": %.1f}\n",
               c.mode ? "mix" : "read", c.pf, c.pf_hint ? "evict_first" : "none", c.load_first ? "evict_first" : "evict_normal",
               best, tot / reps, rd / (best * 1e-3) / 1e9, bytes / (best * 1e-3) / 1e9);
    }
    cudaFree(x); cudaFree(q); cudaFree(sc); cudaFree(zp);
    return 0;
}
