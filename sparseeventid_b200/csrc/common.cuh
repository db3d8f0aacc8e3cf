// Shared device helpers for libscn_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/scn_b200.h"

// number of kernels of THIS library launched so far (library kernels such as CUB's are not counted)
extern unsigned long long g_scn_launch_count;
#define SCN_LAUNCH_CHECK()                                \
  do {                                                    \
    ++g_scn_launch_count;                                 \
    cudaError_t e__ = cudaGetLastError();                 \
    if (e__ != cudaSuccess) return (int)e__;              \
  } while (0)
#define SCN_CUDA(x)                                       \
  do {                                                    \
    cudaError_t e__ = (x);                                \
    if (e__ != cudaSuccess) return (int)e__;              \
  } while (0)

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------------------
// A training step is ~830 dependent launches; between two of them the GPU drains the first grid, flushes, and only then
// starts scheduling the second (~2-3 us each).  The hot-path kernels are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization: a kernel signals griddepcontrol.launch_dependents as its first
// instruction, so the NEXT kernel's CTAs are scheduled onto SMs as this one's CTAs retire and run their prologue
// (barrier init, TMEM allocation, coefficient loads from parameters) early; every kernel executes griddepcontrol.wait
// -- all prerequisite grids complete and their memory visible -- BEFORE its first access to global memory that a
// preceding kernel may have written or may still read, so results do not change.  A dependent grid is only launched
// once every CTA of its primary has started, so a waiting CTA never starves the grid it waits for.  The instructions
// are no-ops for a kernel launched the ordinary way.
#include <utility>
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
template <typename... KArgs, typename... Args>
inline cudaError_t scn_launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

static constexpr uint64_t kEmptyKey = ~0ull;
static constexpr int kNumSMs = 148;   // B200: 2 dies x 74 SMs

__host__ __device__ inline int64_t round_up_i64(int64_t a, int64_t b) { return (a + b - 1) / b * b; }
static inline unsigned grid_for(int64_t work, int block) {
  int64_t g = (work + block - 1) / block;
  if (g < 1) g = 1;
  return (unsigned)g;
}

// ---- feature element access: fp32 or bf16 storage, fp32 math ------------------------------
template <typename T> struct Elem;
template <> struct Elem<float> {
  static __device__ __forceinline__ float ld(const float* p) { return *p; }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
};
template <> struct Elem<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

// 4 consecutive elements <-> float4 (16-byte fp32 / 8-byte bf16 transactions)
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float4 ld4(const __nv_bfloat16* p) {
  uint2 u = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&u.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&u.y);
  float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ void st4(__nv_bfloat16* p, float4 v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
  __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&a);
  u.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = u;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// ---- packed site keys: batch:16 | x0:16 | x1:16 | x2:16 ----------------------------------
__host__ __device__ __forceinline__ uint64_t key_pack(int x0, int x1, int x2, int b) {
  return ((uint64_t)(uint16_t)b << 48) | ((uint64_t)(uint16_t)x0 << 32) | ((uint64_t)(uint16_t)x1 << 16) |
         (uint64_t)(uint16_t)x2;
}
__host__ __device__ __forceinline__ void key_unpack(uint64_t k, int& x0, int& x1, int& x2, int& b) {
  b = (int)(k >> 48);
  x0 = (int)((k >> 32) & 0xFFFF);
  x1 = (int)((k >> 16) & 0xFFFF);
  x2 = (int)(k & 0xFFFF);
}

// ---- hashing: murmur3 finaliser, buckets of 8 slots ---------------------------------------
__device__ __forceinline__ uint32_t key_hash(uint64_t k) {
  k ^= k >> 33;
  k *= 0xff51afd7ed558ccdULL;
  k ^= k >> 33;
  k *= 0xc4ceb9fe1a85ec53ULL;
  k ^= k >> 33;
  return (uint32_t)k;
}

// Cooperative lookup by a group of 8 consecutive lanes (all 32 lanes of the warp must call;
// `active` false lanes/groups idle but take part in the warp-wide ballots).
// Returns the value for `key` or -1.  One probe step reads one 64-byte bucket per group.
__device__ __forceinline__ int hash_lookup_group8(const uint64_t* __restrict__ tk, const int32_t* __restrict__ tv,
                                                  uint32_t bucket_mask, uint64_t key, bool active) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned sub = lane & 7u;
  const unsigned gshift = lane & 24u;
  uint32_t bucket = key_hash(key) & bucket_mask;
  int result = -1;
  bool done = !active;
  while (__any_sync(0xffffffffu, !done)) {
    uint64_t k = done ? kEmptyKey : tk[(size_t)bucket * 8 + sub];
    unsigned hit = (__ballot_sync(0xffffffffu, !done && k == key) >> gshift) & 0xffu;
    unsigned emp = (__ballot_sync(0xffffffffu, !done && k == kEmptyKey) >> gshift) & 0xffu;
    if (!done) {
      if (hit) {
        int slot = __ffs(hit) - 1;
        result = tv[(size_t)bucket * 8 + slot];
        done = true;
      } else if (emp) {
        done = true;
      } else {
        bucket = (bucket + 1) & bucket_mask;
      }
    }
  }
  return result;
}

// Same lookup with 4 lanes per query: each lane reads two adjacent slots (one 16-byte load), so a query still costs
// one 64-byte bucket per probe step but only half the threads.  Used by the submanifold rulebook builder.
__device__ __forceinline__ int hash_lookup_group4(const uint64_t* __restrict__ tk, const int32_t* __restrict__ tv,
                                                  uint32_t bucket_mask, uint64_t key, bool active) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned sub = lane & 3u;
  const unsigned gshift = lane & 28u;
  uint32_t bucket = key_hash(key) & bucket_mask;
  int result = -1;
  bool done = !active;
  while (__any_sync(0xffffffffu, !done)) {
    ulonglong2 k2 = make_ulonglong2(kEmptyKey, kEmptyKey);
    if (!done) k2 = *reinterpret_cast<const ulonglong2*>(tk + (size_t)bucket * 8 + sub * 2);
    const unsigned h0 = (__ballot_sync(0xffffffffu, !done && k2.x == key) >> gshift) & 0xfu;
    const unsigned h1 = (__ballot_sync(0xffffffffu, !done && k2.y == key) >> gshift) & 0xfu;
    const unsigned em = (__ballot_sync(0xffffffffu, !done && (k2.x == kEmptyKey || k2.y == kEmptyKey)) >> gshift) & 0xfu;
    if (!done) {
      if (h0 | h1) {
        const int slot = h0 ? (__ffs(h0) - 1) * 2 : (__ffs(h1) - 1) * 2 + 1;
        result = tv[(size_t)bucket * 8 + slot];
        done = true;
      } else if (em) {
        done = true;
      } else {
        bucket = (bucket + 1) & bucket_mask;
      }
    }
  }
  return result;
}
