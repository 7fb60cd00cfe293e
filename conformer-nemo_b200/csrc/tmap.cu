// cuTensorMapEncodeTiled without linking libcuda: the entry point is resolved through the CUDA runtime, so the
// shared library loads (and exports its symbols) on a machine that has no driver installed.
#include <string.h>

#include <mutex>
#include <unordered_map>

#include "common.cuh"

namespace cfb {

namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
std::once_flag g_once;

void resolve() {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) g_encode = reinterpret_cast<EncodeTiledFn>(fn);
}
}  // namespace

bool encode_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                      const uint64_t* strides_bytes, const uint32_t* box, std::string* err) {
  return encode_tmap(map, base, false, rank, dims, strides_bytes, box, err);
}

bool encode_tmap(CUtensorMap* map, const void* base, bool is_f32, int rank, const uint64_t* dims,
                 const uint64_t* strides_bytes, const uint32_t* box, std::string* err) {
  return encode_tmap_ex(map, base, is_f32, rank, dims, strides_bytes, box, true, err);
}

bool encode_tmap_ex(CUtensorMap* map, const void* base, bool is_f32, int rank, const uint64_t* dims,
                    const uint64_t* strides_bytes, const uint32_t* box, bool swizzle128, std::string* err) {
  // A forward pass re-encodes the same few hundred descriptors on every call (same workspace, same shapes); the
  // driver call costs ~1-2 us each, which is visible at 260 launches per forward.  Per-thread cache, no locking.
  struct Key {
    const void* base;
    uint64_t dims[5], strides[4];
    uint32_t box[5];
    int rank, f32;
    bool operator==(const Key& o) const { return memcmp(this, &o, sizeof(Key)) == 0; }
  };
  struct KeyHash {
    size_t operator()(const Key& k) const {
      const uint64_t* w = reinterpret_cast<const uint64_t*>(&k);
      uint64_t hsh = 1469598103934665603ull;
      for (size_t i = 0; i < sizeof(Key) / 8; ++i) hsh = (hsh ^ w[i]) * 1099511628211ull;
      return static_cast<size_t>(hsh);
    }
  };
  static_assert(sizeof(Key) % 8 == 0, "Key is hashed as 64-bit words");
  thread_local std::unordered_map<Key, CUtensorMap, KeyHash> cache;
  Key key;
  memset(&key, 0, sizeof(key));
  key.base = base;
  key.rank = rank;
  key.f32 = (is_f32 ? 1 : 0) | (swizzle128 ? 0 : 2);
  for (int i = 0; i < rank; ++i) {
    key.dims[i] = dims[i];
    key.box[i] = box[i];
    if (i + 1 < rank) key.strides[i] = strides_bytes[i];
  }
  auto hit = cache.find(key);
  if (hit != cache.end()) {
    *map = hit->second;
    return true;
  }
  std::call_once(g_once, resolve);
  if (g_encode == nullptr) {
    if (err) *err = "cuTensorMapEncodeTiled is not available (no CUDA driver?)";
    return false;
  }
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bdim[5];
  cuuint32_t estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = 1;
    if (i + 1 < rank) gstr[i] = strides_bytes[i];
  }
  CUresult r = g_encode(map, is_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, static_cast<cuuint32_t>(rank), const_cast<void*>(base),
                        gdim, gstr, bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    if (err) {
      char buf[256];
      snprintf(buf, sizeof(buf),
               "cuTensorMapEncodeTiled failed (CUresult %d) rank=%d dims=[%llu,%llu,..] stride0=%llu box=[%u,%u,..] base=%p",
               static_cast<int>(r), rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
               (unsigned long long)(rank > 1 ? strides_bytes[0] : 0), box[0], rank > 1 ? box[1] : 0, base);
      *err = buf;
    }
    return false;
  }
  if (cache.size() > 8192) cache.clear();
  cache.emplace(key, *map);
  return true;
}

namespace {
thread_local int g_pdl_auto = 0;  // set by the engine per forward (small batches), see set_pdl_auto
}
// Programmatic dependent launch.  Measured on cfg2 (r01q): 8.65 ms/step with PDL vs 8.53 without under CUDA-graph replay,
// 8.84 vs 8.99 eager -- at full size launch gaps are not what separates the kernel sum from the step time.  For SMALL
// batches they are: an 8-GPU share of cfg3 (~3000 token rows, every kernel a fraction of a wave) runs 2.93 -> 2.86 ms
// (r5b).  So the engine turns it on per forward below a row count.
bool pdl_enabled() { return g_pdl_auto != 0; }
void set_pdl_auto(bool on) { g_pdl_auto = on ? 1 : 0; }

}  // namespace cfb
