// Host-side helpers shared by every launcher: the tensor-map encoder (with a cache), the per-device
// dynamic-shared-memory attribute, the SM count.
#include "common.cuh"

#include <cstring>
#include <mutex>
#include <unordered_map>

namespace quanta {

EncodeTiledFn get_encode_tiled() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            return nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// cuTensorMapEncodeTiled is a pure function of its arguments and costs ~1-2 us of host time; the hot entries
// are called again and again on the same weights (a linear layer's forward), so the encoded maps are kept in
// a small cache keyed on every argument (bounded: cleared when it reaches 4096 entries).
namespace {
struct MapKey {
    uint64_t base, inner, outer, pitch;
    uint32_t box_inner, box_outer;
    int dtype, swizzle;
    bool operator==(const MapKey& o) const { return std::memcmp(this, &o, sizeof(MapKey)) == 0; }
};
struct MapKeyHash {
    size_t operator()(const MapKey& k) const {
        uint64_t h = 1469598103934665603ull;
        const uint64_t w[6] = {k.base, k.inner, k.outer, k.pitch, ((uint64_t)k.box_inner << 32) | k.box_outer,
                               ((uint64_t)(uint32_t)k.dtype << 32) | (uint32_t)k.swizzle};
        for (uint64_t v : w) { h ^= v; h *= 1099511628211ull; }
        return (size_t)h;
    }
};
std::mutex g_map_mutex;
std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_map_cache;
}  // namespace

int make_tensor_map_2d(CUtensorMap* map, CUtensorMapDataType dtype, size_t elem_bytes, const void* base,
                       uint64_t inner, uint64_t outer, uint64_t pitch_bytes, uint32_t box_inner,
                       uint32_t box_outer, CUtensorMapSwizzle swizzle) {
    EncodeTiledFn enc = get_encode_tiled();
    if (!enc) return QUANTA_EDRIVER;
    (void)elem_bytes;
    MapKey key;
    std::memset(&key, 0, sizeof(key));
    key.base = reinterpret_cast<uint64_t>(base); key.inner = inner; key.outer = outer; key.pitch = pitch_bytes;
    key.box_inner = box_inner; key.box_outer = box_outer; key.dtype = (int)dtype; key.swizzle = (int)swizzle;
    {
        std::lock_guard<std::mutex> lock(g_map_mutex);
        auto it = g_map_cache.find(key);
        if (it != g_map_cache.end()) { *map = it->second; return QUANTA_OK; }
    }
    cuuint64_t dims[2] = {inner, outer};
    cuuint64_t strides[1] = {pitch_bytes};
    cuuint32_t box[2] = {box_inner, box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, dtype, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return QUANTA_EDRIVER;
    {
        std::lock_guard<std::mutex> lock(g_map_mutex);
        if (g_map_cache.size() >= 4096) g_map_cache.clear();
        g_map_cache.emplace(key, *map);
    }
    return QUANTA_OK;
}


int ensure_dynamic_smem(const void* func, int bytes) {
    static std::mutex mu;
    static std::unordered_map<uint64_t, int> set;           // (function, device) -> bytes already granted
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    const uint64_t key = reinterpret_cast<uint64_t>(func) * 131u + (uint64_t)(uint32_t)dev;
    std::lock_guard<std::mutex> lock(mu);
    auto it = set.find(key);
    if (it != set.end() && it->second >= bytes) return 0;
    e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return (int)e;
    set[key] = bytes;
    return 0;
}

int device_sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return kNumSMs;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = kNumSMs;
        cached[dev] = n < kNumSMs ? n : kNumSMs;
    }
    return cached[dev];
}

}  // namespace quanta
