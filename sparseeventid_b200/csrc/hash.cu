// Coordinate hash + InputLayer rules.  Replaces SCN's per-sample google::dense_hash_map grids
// (SURVEY.md 2.2 row 1-2; reference call site src/networks/resnet.py:26-29,40-43,143).
// HBM/L2-latency-bound integer work: one 64-byte bucket read per probe step per 8-lane group.
#include <cub/cub.cuh>

#include "common.cuh"

namespace {

// info (optional, int32[4]): [1] |= 1 when a coordinate or batch index does not fit its 16-bit key field (negative, or
// >= 65536 / batch >= 65535: the packed keys of two different sites would alias), [2] = max batch index seen.
template <typename T>
__global__ void k_pack_coords(const T* __restrict__ c, int64_t n, int ncols, int dim, uint64_t* __restrict__ keys,
                              int32_t* __restrict__ info) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int b = 0;
  bool bad = false;
  if (i < n) {
    const T* r = c + i * ncols;
    int x[3] = {0, 0, 0};
    for (int a = 0; a < dim && a < 3; ++a) {
      const long long v = (long long)r[a];
      bad |= v < 0 || v > 65535;
      x[a] = (int)v;
    }
    const long long bv = ncols > dim ? (long long)r[dim] : 0;
    bad |= bv < 0 || bv >= 65535;
    b = (int)bv;
    keys[i] = key_pack(x[0], x[1], x[2], b);
  }
  if (info != nullptr) {
    const int bmax = __reduce_max_sync(0xffffffffu, bad ? 0 : b);
    const bool any_bad = __any_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0) {
      if (any_bad) atomicOr(info + 1, 1);
      if (bmax > 0) atomicMax(info + 2, bmax);
    }
  }
}

__global__ void k_unpack_keys(const uint64_t* __restrict__ keys, int64_t n, int4* __restrict__ out) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  int x0, x1, x2, b;
  key_unpack(keys[i], x0, x1, x2, b);
  out[i] = make_int4(x0, x1, x2, b);
}

// Insert with "smallest value wins" (first appearance).  8 lanes per key.  Returns the slot.
__device__ __forceinline__ int hash_insert_min_group8(uint64_t* tk, int32_t* tv, uint32_t bucket_mask, uint64_t key,
                                                      int val, bool active) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned sub = lane & 7u;
  const unsigned gshift = lane & 24u;
  uint32_t bucket = key_hash(key) & bucket_mask;
  bool done = !active;
  int slot_out = -1;
  while (__any_sync(0xffffffffu, !done)) {
    uint64_t k = done ? 0ull : __ldcg(reinterpret_cast<const unsigned long long*>(tk + (size_t)bucket * 8 + sub));
    unsigned hit = (__ballot_sync(0xffffffffu, !done && k == key) >> gshift) & 0xffu;
    unsigned emp = (__ballot_sync(0xffffffffu, !done && k == kEmptyKey) >> gshift) & 0xffu;
    const bool want_cas = !done && !hit && emp;
    const int eslot = emp ? __ffs(emp) - 1 : 0;
    unsigned long long prev = 0ull;
    if (want_cas && sub == 0)
      prev = atomicCAS(reinterpret_cast<unsigned long long*>(tk + (size_t)bucket * 8 + eslot), kEmptyKey, key);
    prev = __shfl_sync(0xffffffffu, prev, gshift);
    if (!done) {
      if (hit) {
        int slot = __ffs(hit) - 1;
        slot_out = (int)(bucket * 8 + slot);
        if (sub == 0) atomicMin(tv + slot_out, val);
        done = true;
      } else if (emp) {
        if (prev == kEmptyKey || prev == key) {
          slot_out = (int)(bucket * 8 + eslot);
          if (sub == 0) atomicMin(tv + slot_out, val);
          done = true;
        }  // else: lost the race for that slot to another key; re-read the same bucket
      } else {
        bucket = (bucket + 1) & bucket_mask;
      }
    }
  }
  return slot_out;
}

__global__ void k_insert(const uint64_t* __restrict__ keys, int64_t n, uint64_t* tk, int32_t* tv, uint32_t bucket_mask,
                         int32_t* __restrict__ slot_of) {
  pdl_launch_dependents();
  pdl_wait();
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t i = t >> 3;
  bool active = i < n;
  uint64_t key = active ? keys[i] : 0ull;
  int slot = hash_insert_min_group8(tk, tv, bucket_mask, key, (int)i, active);
  if (active && slot_of && (threadIdx.x & 7) == 0) slot_of[i] = slot;
}

__global__ void k_lookup(const uint64_t* __restrict__ q, int64_t n, const uint64_t* __restrict__ tk,
                         const int32_t* __restrict__ tv, uint32_t bucket_mask, int32_t* __restrict__ out) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t i = t >> 3;
  bool active = i < n;
  uint64_t key = active ? q[i] : 0ull;
  int r = hash_lookup_group8(tk, tv, bucket_mask, key, active);
  if (active && (threadIdx.x & 7) == 0) out[i] = r;
}

__global__ void k_first_flag(const int32_t* __restrict__ slot_of, const int32_t* __restrict__ tv, int64_t n,
                             int32_t* __restrict__ flag) {
  pdl_launch_dependents();
  pdl_wait();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) flag[i] = (tv[slot_of[i]] == (int)i) ? 1 : 0;
}

__global__ void k_assign_rows(const uint64_t* __restrict__ keys, const int32_t* __restrict__ slot_of,
                              const int32_t* __restrict__ tv, const int32_t* __restrict__ flag,
                              const int32_t* __restrict__ rank, int64_t n, int32_t* __restrict__ row_of_input,
                              uint64_t* __restrict__ keys_out, int32_t* __restrict__ n_active) {
  pdl_launch_dependents();
  pdl_wait();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  int first = tv[slot_of[i]];
  row_of_input[i] = rank[first];
  if (flag[i]) keys_out[rank[i]] = keys[i];
  if (i == n - 1) *n_active = rank[i] + flag[i];
}

__global__ void k_store_rows(const int32_t* __restrict__ slot_of, const int32_t* __restrict__ flag,
                             const int32_t* __restrict__ rank, int64_t n, int32_t* tv) {
  pdl_launch_dependents();
  pdl_wait();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n && flag[i]) tv[slot_of[i]] = rank[i];
}

size_t scan_temp_bytes(int64_t n) {
  size_t b = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, b, (const int32_t*)nullptr, (int32_t*)nullptr, (int)n);
  return round_up_i64((int64_t)b, 256);
}

}  // namespace

unsigned long long g_scn_launch_count = 0;

extern "C" const char* scn_version(void) { return "scn_b200 0.1 sm_100a"; }
extern "C" uint64_t scn_launch_count(void) { return (uint64_t)g_scn_launch_count; }

extern "C" int64_t scn_hash_capacity(int64_t n) {
  int64_t c = 1024;
  while (c < 2 * n) c <<= 1;
  return c;
}

extern "C" int scn_pack_coords_checked(const void* coords, int coord_dtype, int64_t n, int ncols, int dimension,
                                       uint64_t* keys, int32_t* info, void* stream) {
  if (n == 0) return SCN_OK;
  if (!coords || !keys || dimension < 1 || dimension > 3 || (ncols != dimension && ncols != dimension + 1))
    return SCN_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned g = grid_for(n, 256);
  switch (coord_dtype) {
    case SCN_COORD_I64: k_pack_coords<long long><<<g, 256, 0, s>>>((const long long*)coords, n, ncols, dimension, keys, info); break;
    case SCN_COORD_I32: k_pack_coords<int><<<g, 256, 0, s>>>((const int*)coords, n, ncols, dimension, keys, info); break;
    case SCN_COORD_F32: k_pack_coords<float><<<g, 256, 0, s>>>((const float*)coords, n, ncols, dimension, keys, info); break;
    case SCN_COORD_F64: k_pack_coords<double><<<g, 256, 0, s>>>((const double*)coords, n, ncols, dimension, keys, info); break;
    default: return SCN_ERR_ARG;
  }
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

extern "C" int scn_unpack_keys(const uint64_t* keys, int64_t n, int32_t* coords4, void* stream) {
  if (n == 0) return SCN_OK;
  if (!keys || !coords4) return SCN_ERR_ARG;
  k_unpack_keys<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(keys, n, (int4*)coords4);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

static int clear_table(uint64_t* tk, int32_t* tv, int64_t cap, cudaStream_t s) {
  if (cap < 8 || (cap & (cap - 1))) return SCN_ERR_ARG;
  SCN_CUDA(cudaMemsetAsync(tk, 0xff, (size_t)cap * sizeof(uint64_t), s));
  SCN_CUDA(cudaMemsetAsync(tv, 0x7f, (size_t)cap * sizeof(int32_t), s));
  return SCN_OK;
}

extern "C" int scn_hash_build(const uint64_t* keys, int64_t n, uint64_t* table_keys, int32_t* table_vals,
                              int64_t capacity, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (!table_keys || !table_vals || capacity < 2 * n) return SCN_ERR_ARG;
  int rc = clear_table(table_keys, table_vals, capacity, s);
  if (rc) return rc;
  if (n == 0) return SCN_OK;
  SCN_CUDA(scn_launch_pdl(k_insert, dim3(grid_for(n * 8, 256)), dim3(256), 0, s, keys, n, table_keys, table_vals, (uint32_t)(capacity / 8 - 1), (int32_t*)nullptr));
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

extern "C" int scn_hash_lookup(const uint64_t* queries, int64_t n, const uint64_t* table_keys,
                               const int32_t* table_vals, int64_t capacity, int32_t* out, void* stream) {
  if (n == 0) return SCN_OK;
  if (!queries || !table_keys || !table_vals || !out) return SCN_ERR_ARG;
  k_lookup<<<grid_for(n * 8, 256), 256, 0, (cudaStream_t)stream>>>(queries, n, table_keys, table_vals,
                                                                   (uint32_t)(capacity / 8 - 1), out);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

extern "C" size_t scn_input_rules_workspace(int64_t n) {
  return (size_t)(3 * round_up_i64(n * 4, 256)) + scan_temp_bytes(n) + 256;
}

extern "C" int scn_input_layer_rules(const uint64_t* keys_in, int64_t n, uint64_t* table_keys, int32_t* table_vals,
                                     int64_t capacity, int32_t* row_of_input, uint64_t* keys_out,
                                     int32_t* n_active_dev, void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (!table_keys || !table_vals || !n_active_dev || capacity < 2 * n) return SCN_ERR_ARG;
  int rc = clear_table(table_keys, table_vals, capacity, s);
  if (rc) return rc;
  if (n == 0) {
    SCN_CUDA(cudaMemsetAsync(n_active_dev, 0, sizeof(int32_t), s));
    return SCN_OK;
  }
  if (workspace_bytes < scn_input_rules_workspace(n) || !workspace) return SCN_ERR_WORKSPACE;
  char* w = (char*)workspace;
  size_t seg = (size_t)round_up_i64(n * 4, 256);
  int32_t* slot_of = (int32_t*)w;
  int32_t* flag = (int32_t*)(w + seg);
  int32_t* rank = (int32_t*)(w + 2 * seg);
  void* tmp = w + 3 * seg;
  size_t tmp_bytes = scan_temp_bytes(n);
  uint32_t bm = (uint32_t)(capacity / 8 - 1);
  SCN_CUDA(scn_launch_pdl(k_insert, dim3(grid_for(n * 8, 256)), dim3(256), 0, s, keys_in, n, table_keys, table_vals, bm, slot_of));
  SCN_LAUNCH_CHECK();
  SCN_CUDA(scn_launch_pdl(k_first_flag, dim3(grid_for(n, 256)), dim3(256), 0, s, slot_of, table_vals, n, flag));
  SCN_LAUNCH_CHECK();
  SCN_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, flag, rank, (int)n, s));
  SCN_CUDA(scn_launch_pdl(k_assign_rows, dim3(grid_for(n, 256)), dim3(256), 0, s, keys_in, slot_of, table_vals, flag, rank, n,
                          row_of_input, keys_out, n_active_dev));
  SCN_LAUNCH_CHECK();
  SCN_CUDA(scn_launch_pdl(k_store_rows, dim3(grid_for(n, 256)), dim3(256), 0, s, slot_of, flag, rank, n, table_vals));
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}
