// Rulebook builders on the GPU coordinate hash.  Replace SCN's host-side
// SubmanifoldConvolution_SgToRules and Convolution_InputSgsToRulesAndOutputSgs (SURVEY.md 2.2;
// reference call sites src/networks/sparse_building_blocks.py:29-34,110-117).
// Output: neighbour tables nbr[K][n_pad] (see include/scn_b200.h) + the SCN pair-list form.
#include <cub/cub.cuh>

#include "common.cuh"

namespace {

// One 4-lane group per (half-offset h, site r).  Probes site + d_h; the mirrored entry
// (K-1-h, neighbour) follows from symmetry, so only (K-1)/2 of the K offsets touch the hash.
__global__ void k_subm_probe(const uint64_t* __restrict__ keys, int64_t n, const uint64_t* __restrict__ tk,
                             const int32_t* __restrict__ tv, uint32_t bucket_mask, int f0, int f1, int f2, int K,
                             int32_t* __restrict__ nbr, int64_t n_pad) {
  pdl_launch_dependents();
  pdl_wait();
  const int half = (K - 1) / 2;
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t item = t >> 2;
  bool active = item < (int64_t)half * n;
  int h = 0;
  int64_t r = 0;
  uint64_t qkey = 0;
  if (active) {
    h = (int)(item / n);
    r = item - (int64_t)h * n;
    int x0, x1, x2, b;
    key_unpack(keys[r], x0, x1, x2, b);
    int a2 = h % f2, a1 = (h / f2) % f1, a0 = h / (f2 * f1);
    x0 += a0 - f0 / 2;
    x1 += a1 - f1 / 2;
    x2 += a2 - f2 / 2;
    // coordinates live in 16-bit fields: a step outside [0, 65535] can never be a site and must
    // not borrow into the neighbouring field of the packed key
    active = ((unsigned)x0 < 65536u) && ((unsigned)x1 < 65536u) && ((unsigned)x2 < 65536u);
    qkey = key_pack(x0, x1, x2, b);
  }
  int j = hash_lookup_group4(tk, tv, bucket_mask, qkey, active);
  if (active && (threadIdx.x & 3) == 0 && j >= 0) {
    nbr[(int64_t)h * n_pad + r] = j;
    nbr[(int64_t)(K - 1 - h) * n_pad + j] = (int)r;
  }
}

__global__ void k_identity_rows(int32_t* __restrict__ dst, int64_t n) {
  pdl_launch_dependents();
  pdl_wait();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (int)i;
}

__global__ void k_strided_tables(const int32_t* __restrict__ out_row_of_in, const int32_t* __restrict__ off_of_in,
                                 int64_t n_in, int32_t* __restrict__ down, int64_t n_out_pad,
                                 int32_t* __restrict__ up, int64_t n_in_pad) {
  pdl_launch_dependents();
  pdl_wait();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_in) return;
  int q = out_row_of_in[i], k = off_of_in[i];
  if (down) down[(int64_t)k * n_out_pad + q] = (int)i;
  if (up) up[(int64_t)k * n_in_pad + i] = q;
}

struct ValidFlag {
  const int32_t* nbr;
  __host__ __device__ int32_t operator()(int64_t i) const { return nbr[i] >= 0 ? 1 : 0; }
};

__global__ void k_count_valid(const int32_t* __restrict__ nbr, int64_t n, int64_t n_pad, int32_t* __restrict__ counts) {
  int k = blockIdx.y;
  int c = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    c += nbr[(int64_t)k * n_pad + i] >= 0;
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(counts + k, c);
}

__global__ void k_fill_pairs(const int32_t* __restrict__ nbr, const int32_t* __restrict__ pos, int K, int64_t n_pad,
                             int32_t* __restrict__ pair_in, int32_t* __restrict__ pair_out,
                             int32_t* __restrict__ offsets) {
  int64_t total = (int64_t)K * n_pad;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= total) return;
  int v = nbr[i];
  int p = pos[i];
  int64_t k = i / n_pad, o = i - k * n_pad;
  if (o == 0) offsets[k] = p;
  if (v >= 0) {
    pair_in[p] = v;
    pair_out[p] = (int)o;
  }
  if (i == total - 1) offsets[K] = p + (v >= 0);
}

using ValidIter = cub::TransformInputIterator<int32_t, ValidFlag, cub::CountingInputIterator<int64_t>>;
size_t pairs_scan_temp(int64_t total) {
  size_t b = 0;
  cub::CountingInputIterator<int64_t> cnt(0);
  ValidIter it(cnt, ValidFlag{nullptr});
  cub::DeviceScan::ExclusiveSum(nullptr, b, it, (int32_t*)nullptr, (int)total);
  return (size_t)round_up_i64((int64_t)b, 256);
}
}  // namespace

extern "C" int scn_subm_rulebook(const uint64_t* keys, int64_t n, const uint64_t* table_keys,
                                 const int32_t* table_vals, int64_t capacity, int f0, int f1, int f2, int32_t* nbr,
                                 int64_t n_pad, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (f0 < 1 || f1 < 1 || f2 < 1 || !(f0 & 1) || !(f1 & 1) || !(f2 & 1)) return SCN_ERR_ARG;
  if (n_pad < n || (n_pad & 127)) return SCN_ERR_ARG;
  const int K = f0 * f1 * f2;
  if (n_pad == 0) return SCN_OK;
  if (!nbr) return SCN_ERR_ARG;
  SCN_CUDA(cudaMemsetAsync(nbr, 0xff, (size_t)K * n_pad * sizeof(int32_t), s));
  if (n == 0) return SCN_OK;
  if (!keys || !table_keys || !table_vals) return SCN_ERR_ARG;
  const int half = (K - 1) / 2;
  SCN_CUDA(scn_launch_pdl(k_identity_rows, dim3(grid_for(n, 256)), dim3(256), 0, s, nbr + (int64_t)half * n_pad, n));
  SCN_LAUNCH_CHECK();
  if (half > 0) {
    SCN_CUDA(scn_launch_pdl(k_subm_probe, dim3(grid_for((int64_t)half * n * 4, 256)), dim3(256), 0, s, keys, n, table_keys,
                            table_vals, (uint32_t)(capacity / 8 - 1), f0, f1, f2, K, nbr, n_pad));
    SCN_LAUNCH_CHECK();
  }
  return SCN_OK;
}

// ---- strided rulebook (filter == stride) through the coordinate hash ------------------------------------------------
// Output sites are the distinct coarse keys; they are found and NUMBERED IN FIRST-APPEARANCE ORDER over the input rows
// by the InputLayer machinery (hash insert with smallest-index-wins, flag, scan), which is SparseConvNet's own order
// (output rows are created on first touch) and leaves behind the coarse level's hash table, so the next level needs no
// separate build.  A 64-bit radix sort of the coarse keys costs 8 onesweep passes per level (~135 us even for 7 k sites).
namespace {
__global__ void k_coarse_keys_off(const uint64_t* __restrict__ keys, int64_t n, int s0, int s1, int s2,
                                  uint64_t* __restrict__ qkeys, int32_t* __restrict__ off) {
  pdl_launch_dependents();
  pdl_wait();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  int x0, x1, x2, b;
  key_unpack(keys[i], x0, x1, x2, b);
  int q0 = x0 / s0, q1 = x1 / s1, q2 = x2 / s2;
  qkeys[i] = key_pack(q0, q1, q2, b);
  off[i] = ((x0 - q0 * s0) * s1 + (x1 - q1 * s1)) * s2 + (x2 - q2 * s2);
}
}  // namespace

extern "C" size_t scn_strided_hash_workspace(int64_t n) {
  return (size_t)round_up_i64(n * 8, 256) + scn_input_rules_workspace(n) + 256;
}

extern "C" int scn_strided_rulebook_hash(const uint64_t* keys_in, int64_t n, int s0, int s1, int s2, uint64_t* table_keys,
                                         int32_t* table_vals, int64_t capacity, uint64_t* keys_out,
                                         int32_t* out_row_of_in, int32_t* off_of_in, int32_t* n_out_dev, void* workspace,
                                         size_t workspace_bytes, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (s0 < 1 || s1 < 1 || s2 < 1 || !n_out_dev || !table_keys || !table_vals) return SCN_ERR_ARG;
  if (n > 0 && (!workspace || workspace_bytes < scn_strided_hash_workspace(n))) return SCN_ERR_WORKSPACE;
  uint64_t* qkeys = (uint64_t*)workspace;
  char* ws2 = (char*)workspace + round_up_i64(n * 8, 256);
  if (n > 0) {
    SCN_CUDA(scn_launch_pdl(k_coarse_keys_off, dim3(grid_for(n, 256)), dim3(256), 0, s, keys_in, n, s0, s1, s2, qkeys, off_of_in));
    SCN_LAUNCH_CHECK();
  }
  return scn_input_layer_rules(qkeys, n, table_keys, table_vals, capacity, out_row_of_in, keys_out, n_out_dev, ws2,
                               n > 0 ? workspace_bytes - (size_t)round_up_i64(n * 8, 256) : 0, stream);
}

extern "C" int scn_strided_tables(const int32_t* out_row_of_in, const int32_t* off_of_in, int64_t n_in, int K,
                                  int32_t* nbr_down, int64_t n_out_pad, int32_t* nbr_up, int64_t n_in_pad,
                                  void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (K < 1) return SCN_ERR_ARG;
  if (nbr_down && n_out_pad) SCN_CUDA(cudaMemsetAsync(nbr_down, 0xff, (size_t)K * n_out_pad * sizeof(int32_t), s));
  if (nbr_up && n_in_pad) SCN_CUDA(cudaMemsetAsync(nbr_up, 0xff, (size_t)K * n_in_pad * sizeof(int32_t), s));
  if (n_in == 0) return SCN_OK;
  SCN_CUDA(scn_launch_pdl(k_strided_tables, dim3(grid_for(n_in, 256)), dim3(256), 0, s, out_row_of_in, off_of_in, n_in, nbr_down,
                          n_out_pad, nbr_up, n_in_pad));
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

extern "C" size_t scn_rulebook_workspace(int K, int64_t n_pad) {
  int64_t total = (int64_t)K * n_pad;
  return (size_t)round_up_i64(total * 4, 256) + pairs_scan_temp(total) + 256;
}

extern "C" int scn_rulebook_count(const int32_t* nbr, int K, int64_t n, int64_t n_pad, int32_t* counts_dev,
                                  void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (!counts_dev || K < 1) return SCN_ERR_ARG;
  SCN_CUDA(cudaMemsetAsync(counts_dev, 0, (size_t)K * sizeof(int32_t), s));
  if (n == 0) return SCN_OK;
  dim3 g((unsigned)((n + 1023) / 1024 < 1024 ? (n + 1023) / 1024 : 1024), (unsigned)K);
  k_count_valid<<<g, 256, 0, s>>>(nbr, n, n_pad, counts_dev);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

extern "C" int scn_rulebook_pairs(const int32_t* nbr, int K, int64_t n, int64_t n_pad, int32_t* pair_in,
                                  int32_t* pair_out, int32_t* offsets_dev, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  (void)n;
  if (!offsets_dev || K < 1) return SCN_ERR_ARG;
  int64_t total = (int64_t)K * n_pad;
  if (total == 0) {
    SCN_CUDA(cudaMemsetAsync(offsets_dev, 0, (size_t)(K + 1) * sizeof(int32_t), s));
    return SCN_OK;
  }
  if (total > 0x7fffffffLL) return SCN_ERR_UNSUPPORTED;
  if (!workspace || workspace_bytes < scn_rulebook_workspace(K, n_pad)) return SCN_ERR_WORKSPACE;
  int32_t* pos = (int32_t*)workspace;
  void* tmp = (char*)workspace + round_up_i64(total * 4, 256);
  size_t tmp_bytes = pairs_scan_temp(total);
  cub::CountingInputIterator<int64_t> cnt(0);
  ValidIter it(cnt, ValidFlag{nbr});
  SCN_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, it, pos, (int)total, s));
  k_fill_pairs<<<grid_for(total, 256), 256, 0, s>>>(nbr, pos, K, n_pad, pair_in, pair_out, offsets_dev);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}
