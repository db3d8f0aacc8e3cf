// Bandwidth-bound layers: BatchNormalization(+leaky), LeakyReLU, AddTable, InputLayer/OutputLayer
// feature movement, SparseToDense.  Replace SCN's BatchNormalization.cu / LeakyReLU.cu /
// IOLayers.cu / SparseToDense.cu (SURVEY.md 2.2; reference call sites
// src/networks/sparse_building_blocks.py:39,45,80-82,96-98,122,128; src/networks/resnet.py:123-125,143).
// All kernels are HBM-bound: 16-byte (fp32) / 8-byte (bf16) vector accesses along channels,
// fp32 math, column reductions finished with fp64 atomics.
#include <map>
#include <mutex>
#include <type_traits>
#include <utility>

#include "common.cuh"

namespace {

constexpr int kRedThreads = 256;
constexpr int kRedRows = 256;   // rows per block in column reductions

// ---------------------------------------------------------------------------------------------
// Column reductions over [n, C]: each thread owns VEC adjacent channels and strides over rows.
// F::eval(row, c0, out_a[VEC], out_b[VEC]) yields the two per-element quantities to be summed.
// A row has C / VEC channel groups; blockIdx.y selects a slice of CV <= 256 of them (the last slice may hold fewer),
// so any C works: a block covers kRedRows rows of one slice.
// ---------------------------------------------------------------------------------------------
template <int VEC, typename F>
__global__ void __launch_bounds__(kRedThreads) k_col_reduce2(F f, int64_t n, int C, int CV,
                                                             double* __restrict__ acc /*[2][C]*/) {
  extern __shared__ float sred[];   // [RY][CV][2*VEC]
  const int RY = kRedThreads / CV;
  const int g0 = blockIdx.y * CV;                      // first channel group of this slice
  const int ncv = C / VEC - g0 < CV ? C / VEC - g0 : CV;
  const int tx = threadIdx.x % CV, ty = threadIdx.x / CV;
  float a[VEC], b[VEC];
#pragma unroll
  for (int v = 0; v < VEC; ++v) a[v] = b[v] = 0.f;
  const int64_t r0 = (int64_t)blockIdx.x * kRedRows;
  const int64_t r1 = r0 + kRedRows < n ? r0 + kRedRows : n;
  if (ty < RY && tx < ncv) {
    for (int64_t r = r0 + ty; r < r1; r += RY) {
      float va[VEC], vb[VEC];
      f.eval(r, (g0 + tx) * VEC, va, vb);
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        a[v] += va[v];
        b[v] += vb[v];
      }
    }
    float* dst = sred + ((size_t)ty * CV + tx) * 2 * VEC;
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      dst[v] = a[v];
      dst[VEC + v] = b[v];
    }
  }
  __syncthreads();
  // first ncv*VEC*2 threads (looped) sum over ty and publish
  for (int i = threadIdx.x; i < ncv * 2 * VEC; i += kRedThreads) {
    int cx = i / (2 * VEC), w = i % (2 * VEC);
    float s = 0.f;
    for (int y = 0; y < RY; ++y) s += sred[((size_t)y * CV + cx) * 2 * VEC + w];
    int which = w / VEC, c = (g0 + cx) * VEC + (w % VEC);
    if (F::kTwo || which == 0) atomicAdd(acc + (size_t)which * C + c, (double)s);
  }
}

template <typename T, int VEC> struct LoadVec;
template <typename T> struct LoadVec<T, 4> {
  static __device__ __forceinline__ void ld(const T* p, float* o) {
    float4 v = ld4(p);
    o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
  }
  static __device__ __forceinline__ void st(T* p, const float* o) { st4(p, make_float4(o[0], o[1], o[2], o[3])); }
};
// 8 consecutive elements: ONE 16-byte access for bf16 (two for fp32) -- twice the bytes in flight per thread
template <> struct LoadVec<__nv_bfloat16, 8> {
  static __device__ __forceinline__ void ld(const __nv_bfloat16* p, float* o) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[i]));
      o[2 * i] = f.x;
      o[2 * i + 1] = f.y;
    }
  }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, const float* o) {
    uint4 u;
    u.x = pack_bf16x2(o[0], o[1]); u.y = pack_bf16x2(o[2], o[3]);
    u.z = pack_bf16x2(o[4], o[5]); u.w = pack_bf16x2(o[6], o[7]);
    *reinterpret_cast<uint4*>(p) = u;
  }
};
template <> struct LoadVec<float, 8> {
  static __device__ __forceinline__ void ld(const float* p, float* o) {
    const float4 a = ld4(p), b = ld4(p + 4);
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
  }
  static __device__ __forceinline__ void st(float* p, const float* o) {
    st4(p, make_float4(o[0], o[1], o[2], o[3]));
    st4(p + 4, make_float4(o[4], o[5], o[6], o[7]));
  }
};
template <typename T> struct LoadVec<T, 1> {
  static __device__ __forceinline__ void ld(const T* p, float* o) { o[0] = Elem<T>::ld(p); }
  static __device__ __forceinline__ void st(T* p, const float* o) { Elem<T>::st(p, o[0]); }
};

// sum and sum of squares of (x - pivot), pivot = row 0 (kills the cancellation in E[x^2]-E[x]^2)
template <typename T, int VEC> struct StatsF {
  static constexpr bool kTwo = true;
  const T* x; int C;
  __device__ __forceinline__ void eval(int64_t r, int c0, float* a, float* b) const {
    float v[VEC], p[VEC];
    LoadVec<T, VEC>::ld(x + r * C + c0, v);
    LoadVec<T, VEC>::ld(x + c0, p);
#pragma unroll
    for (int i = 0; i < VEC; ++i) { float d = v[i] - p[i]; a[i] = d; b[i] = d * d; }
  }
};
template <typename T, int VEC> struct SumF {
  static constexpr bool kTwo = false;
  const T* x; int C;
  __device__ __forceinline__ void eval(int64_t r, int c0, float* a, float* b) const {
    LoadVec<T, VEC>::ld(x + r * C + c0, a);
#pragma unroll
    for (int i = 0; i < VEC; ++i) b[i] = 0.f;
  }
};
// BN backward sums: d = dout * (y > 0 ? 1 : leak), a = d, b = d * xhat
template <typename T, int VEC> struct BnBwdF {
  static constexpr bool kTwo = true;
  const T* x; const T* dout; const float* mean; const float* invstd; const float* gamma; const float* beta;
  float leak; int C;
  __device__ __forceinline__ void eval(int64_t r, int c0, float* a, float* b) const {
    float v[VEC], d[VEC];
    LoadVec<T, VEC>::ld(x + r * C + c0, v);
    LoadVec<T, VEC>::ld(dout + r * C + c0, d);
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      int c = c0 + i;
      float xh = (v[i] - mean[c]) * invstd[c];
      float y = xh * (gamma ? gamma[c] : 1.f) + (beta ? beta[c] : 0.f);
      float dd = (leak != 1.f && !(y > 0.f)) ? d[i] * leak : d[i];
      a[i] = dd;
      b[i] = dd * xh;
    }
  }
};

template <typename T>
__global__ void k_bn_finalize(const double* __restrict__ acc, const T* __restrict__ x, int64_t n, int C, int training,
                              float eps, float momentum, float* running_mean, float* running_var,
                              float* __restrict__ save_mean, float* __restrict__ save_invstd) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  if (training) {
    double mean = 0.0, var = 0.0;
    if (n > 0) {
      double pivot = (double)Elem<T>::ld(x + c);
      double s1 = acc[c] / (double)n, s2 = acc[C + c] / (double)n;
      mean = pivot + s1;
      var = s2 - s1 * s1;
      if (var < 0.0) var = 0.0;
    }
    double unbiased = var * (double)n / (double)(n > 1 ? n - 1 : 1);   // divisor max(N-1, 1)
    running_mean[c] = (float)((double)momentum * running_mean[c] + (1.0 - (double)momentum) * mean);
    running_var[c] = (float)((double)momentum * running_var[c] + (1.0 - (double)momentum) * unbiased);
    save_mean[c] = (float)mean;
    save_invstd[c] = (float)(1.0 / sqrt(var + (double)eps));
  } else {
    save_mean[c] = running_mean[c];
    save_invstd[c] = (float)(1.0 / sqrt((double)running_var[c] + (double)eps));
  }
}

template <typename T, int VEC>
__global__ void k_bn_apply(const T* __restrict__ x, int64_t nvec, int C, const float* __restrict__ mean,
                           const float* __restrict__ invstd, const float* __restrict__ gamma,
                           const float* __restrict__ beta, float leak, T* __restrict__ out) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= nvec) return;
  int c0 = (int)((i * VEC) % C);
  float v[VEC];
  LoadVec<T, VEC>::ld(x + i * VEC, v);
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    int c = c0 + k;
    float y = (v[k] - mean[c]) * invstd[c] * (gamma ? gamma[c] : 1.f) + (beta ? beta[c] : 0.f);
    v[k] = (leak != 1.f && !(y > 0.f)) ? y * leak : y;
  }
  LoadVec<T, VEC>::st(out + i * VEC, v);
}

// Row-streaming forms of the two apply kernels (C % 8 == 0, C / 8 <= 256): a thread owns 8 fixed channels, folds
// their per-channel coefficients into registers ONCE and then streams rows with 16-byte accesses.  (The
// element-indexed forms above re-load 4-6 per-channel values for every element: LSU-bound at ~1.7 TB/s.)
template <typename T>
__global__ void __launch_bounds__(256) k_bn_apply_rows(const T* __restrict__ x, int64_t n, int C,
                                                       const float* __restrict__ mean, const float* __restrict__ invstd,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       float leak, T* __restrict__ out) {
  const int CV = C >> 3, RY = 256 / CV;
  const int tx = threadIdx.x % CV, ty = threadIdx.x / CV;
  if (ty >= RY) return;
  float sc[8], sh[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int c = tx * 8 + k;
    sc[k] = invstd[c] * (gamma ? gamma[c] : 1.f);
    sh[k] = (beta ? beta[c] : 0.f) - mean[c] * sc[k];
  }
  for (int64_t r = (int64_t)blockIdx.x * RY + ty; r < n; r += (int64_t)gridDim.x * RY) {
    float v[8];
    LoadVec<T, 8>::ld(x + r * C + tx * 8, v);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      // same association as the element-indexed kernel: ((x - mean) * invstd) * gamma + beta, up to one rounding
      const float y = fmaf(v[k], sc[k], sh[k]);
      v[k] = (leak != 1.f && !(y > 0.f)) ? y * leak : y;
    }
    LoadVec<T, 8>::st(out + r * C + tx * 8, v);
  }
}

template <typename T>
__global__ void __launch_bounds__(256) k_bn_bwd_apply_rows(const T* __restrict__ x, const T* __restrict__ dout, int64_t n,
                                                           int C, const float* __restrict__ mean,
                                                           const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, float leak, int training,
                                                           const double* __restrict__ acc, T* __restrict__ dx) {
  const int CV = C >> 3, RY = 256 / CV;
  const int tx = threadIdx.x % CV, ty = threadIdx.x / CV;
  if (ty >= RY) return;
  float m[8], is[8], g[8], b[8], s1[8], s2[8];
  const float inv_n = n > 0 ? 1.f / (float)n : 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int c = tx * 8 + k;
    m[k] = mean[c]; is[k] = invstd[c];
    g[k] = gamma ? gamma[c] : 1.f;
    b[k] = beta ? beta[c] : 0.f;
    s1[k] = training ? (float)acc[c] * inv_n : 0.f;
    s2[k] = training ? (float)acc[C + c] * inv_n : 0.f;
  }
  for (int64_t r = (int64_t)blockIdx.x * RY + ty; r < n; r += (int64_t)gridDim.x * RY) {
    float v[8], d[8];
    LoadVec<T, 8>::ld(x + r * C + tx * 8, v);
    LoadVec<T, 8>::ld(dout + r * C + tx * 8, d);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float xh = (v[k] - m[k]) * is[k];
      const float y = xh * g[k] + b[k];
      const float dd = (leak != 1.f && !(y > 0.f)) ? d[k] * leak : d[k];
      v[k] = g[k] * is[k] * (dd - s1[k] - xh * s2[k]);
    }
    LoadVec<T, 8>::st(dx + r * C + tx * 8, v);
  }
}

// ---------------------------------------------------------------------------------------------
// Training-mode BatchNormalization as TWO ordinary launches per direction (C % 8 == 0, C <= 2048):
//   statistics kernel: column sums -> one of two sets of fp64 accumulators (zero on entry), nothing else,
//   apply kernel:      every thread folds the statistics of its 8 channels into registers (forward: scale / shift,
//                      block 0 also writes the saved and running statistics; backward: the three coefficients of dx,
//                      block 0 writes dgamma / dbeta), zeroes the OTHER set of accumulators for the next call and
//                      streams the rows.  The backward apply also sums the columns of the dx it stores: that is the
//                      bias gradient of the convolution in front of the BatchNorm (56 column-sum launches and one read
//                      of every dx per step otherwise).
// The four-launch form (memset, column reduction, finalize, apply), which eval mode and the other channel counts use,
// costs ~27 us (forward) / ~40 us (backward) of launch latency and dependency bubbles even on a 7 k-row level, more than
// the data movement of every level below the first two.  A single cooperative launch per direction (column sums, grid
// barrier, apply, grid barrier, re-zeroing) was measured too and removed (ncu, 495 k rows x 32 channels, backward): 18%
// of the kernel was its final grid barrier + re-zeroing, 7% the first barrier, 102 registers held it to 2 blocks per SM,
// a cooperative launch costs ~6-10 us more than an ordinary one on the stream, and every thread folded the statistics of
// its channels with fp64 divisions and square roots (~6 us per block on the thin fp64 pipe).  Here the kernels run at
// 3-4 blocks x 256 threads per SM with 64 B in flight per thread; the fold is 2 fp64 multiplies, one fma and a
// Newton-refined rsqrt per channel.
// ---------------------------------------------------------------------------------------------
template <typename T> struct Raw8;                       // 8 consecutive elements, kept packed while in flight
template <> struct Raw8<__nv_bfloat16> {
  uint4 u;
  __device__ __forceinline__ void ld(const __nv_bfloat16* p) { u = *reinterpret_cast<const uint4*>(p); }
  __device__ __forceinline__ void get(float* o) const {
    o[0] = __uint_as_float(u.x << 16); o[1] = __uint_as_float(u.x & 0xffff0000u);
    o[2] = __uint_as_float(u.y << 16); o[3] = __uint_as_float(u.y & 0xffff0000u);
    o[4] = __uint_as_float(u.z << 16); o[5] = __uint_as_float(u.z & 0xffff0000u);
    o[6] = __uint_as_float(u.w << 16); o[7] = __uint_as_float(u.w & 0xffff0000u);
  }
};
template <> struct Raw8<float> {
  float4 a, b;
  __device__ __forceinline__ void ld(const float* p) { a = ld4(p); b = ld4(p + 4); }
  __device__ __forceinline__ void get(float* o) const {
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
  }
};
// store 8 values and add what was STORED (after rounding to T) to cs[8]
__device__ __forceinline__ void store8_sum(__nv_bfloat16* p, const float* v, float* cs) {
  Raw8<__nv_bfloat16> r;
  r.u.x = pack_bf16x2(v[0], v[1]); r.u.y = pack_bf16x2(v[2], v[3]);
  r.u.z = pack_bf16x2(v[4], v[5]); r.u.w = pack_bf16x2(v[6], v[7]);
  *reinterpret_cast<uint4*>(p) = r.u;
  float f[8];
  r.get(f);
#pragma unroll
  for (int k = 0; k < 8; ++k) cs[k] += f[k];
}
__device__ __forceinline__ void store8_sum(float* p, const float* v, float* cs) {
  LoadVec<float, 8>::st(p, v);
#pragma unroll
  for (int k = 0; k < 8; ++k) cs[k] += v[k];
}

// Per-thread partial sums a[8] (and b[8] when TWO) (thread = row slot ty x channel group tx) -> acc[c] += sum a,
// acc[C + c] += sum b.  When the channel groups of a row divide a warp (C = 32, 64, 128, 256) lanes that own the same
// channels are summed with shuffles first and only one partial per warp goes through shared memory; otherwise one
// partial per row slot (RY <= 21 then).  sred: 256 x 16 floats.
template <bool TWO>
__device__ __forceinline__ void block_col_sums(float* a, float* b, int C, int CV, int RY, int tx, int ty, bool active,
                                               float* sred, double* acc) {
  constexpr int W = TWO ? 16 : 8;
  int parts;
  if ((32 % CV) == 0) {
    for (int m = CV; m < 32; m <<= 1) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        a[k] += __shfl_xor_sync(0xffffffffu, a[k], m);
        if (TWO) b[k] += __shfl_xor_sync(0xffffffffu, b[k], m);
      }
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane < CV) {
      float* dst = sred + ((size_t)w * CV + tx) * W;
#pragma unroll
      for (int k = 0; k < 8; ++k) { dst[k] = a[k]; if (TWO) dst[8 + k] = b[k]; }
    }
    parts = 8;
  } else {
    if (active) {
      float* dst = sred + ((size_t)ty * CV + tx) * W;
#pragma unroll
      for (int k = 0; k < 8; ++k) { dst[k] = a[k]; if (TWO) dst[8 + k] = b[k]; }
    }
    parts = RY;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < CV * W; i += 256) {
    const int cx = i / W, w = i % W;
    float sum = 0.f;
    for (int y = 0; y < parts; ++y) sum += sred[((size_t)y * CV + cx) * W + w];
    atomicAdd(acc + (size_t)(w >> 3) * C + cx * 8 + (w & 7), (double)sum);
  }
}

// true in every thread of the LAST block of the grid to get here; that block then sees every block's atomics
__device__ __forceinline__ bool last_block(unsigned* ticket) {
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last) __threadfence();
  return last;
}

// Two sets of accumulators, used alternately (BN call i of a stream uses set i & 1): the apply kernel of call i zeroes
// the OTHER set -- nobody reads or writes it while that kernel runs -- so the statistics kernel needs no "last block
// zeroes / finalises" tail (threadfence + ticket + a serial block: ~3 us of a ~8 us kernel on the deep levels) and the
// statistics are folded per thread in the apply kernel: two fp64 multiplies, one fp64 fma and a Newton-refined
// rsqrt per channel (no fp64 division or square root: those made the per-thread fold ~6 us per block).
__device__ __forceinline__ float inv_sqrt_refined(double v) {
  const float r = rsqrtf((float)v);
  const double rd = (double)r;
  return (float)(rd * (1.5 - 0.5 * v * rd * rd));       // one Newton step in fp64: correct to fp32 rounding
}

template <typename T>
__global__ void __launch_bounds__(256, 4) k_bn_stats2(const T* __restrict__ x, int64_t n, int C, double* acc) {
  __shared__ float sred[256 * 16];
  pdl_launch_dependents();
  pdl_wait();
  const int CV = C >> 3, RY = 256 / CV;
  const int tx = threadIdx.x % CV, ty = threadIdx.x / CV;
  const bool active = ty < RY;
  const int64_t stride = (int64_t)gridDim.x * RY;
  float a[8], b[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) a[k] = b[k] = 0.f;
  if (active) {
    float pv[8];
    { Raw8<T> p; p.ld(x + tx * 8); p.get(pv); }          // pivot = row 0 (kills the cancellation in E[x^2] - E[x]^2)
    const T* px = x + tx * 8;
    int64_t r = (int64_t)blockIdx.x * RY + ty;
    for (; r + 3 * stride < n; r += 4 * stride) {
      Raw8<T> v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u].ld(px + (r + u * stride) * C);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float f[8];
        v[u].get(f);
#pragma unroll
        for (int k = 0; k < 8; ++k) { const float d = f[k] - pv[k]; a[k] += d; b[k] = fmaf(d, d, b[k]); }
      }
    }
    for (; r < n; r += stride) {
      Raw8<T> v;
      v.ld(px + r * C);
      float f[8];
      v.get(f);
#pragma unroll
      for (int k = 0; k < 8; ++k) { const float d = f[k] - pv[k]; a[k] += d; b[k] = fmaf(d, d, b[k]); }
    }
  }
  block_col_sums<true>(a, b, C, CV, RY, tx, ty, active, sred, acc);
}

template <typename T>
__global__ void __launch_bounds__(256, 4) k_bn_apply2(const T* __restrict__ x, int64_t n, int C, const float* __restrict__ gamma,
                                                      const float* __restrict__ beta, float* running_mean,
                                                      float* running_var, float eps, float momentum, float leak,
                                                      float* __restrict__ save_mean, float* __restrict__ save_invstd,
                                                      const double* __restrict__ acc, double* __restrict__ acc_other,
                                                      int zero_n, double inv_n, T* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  const int CV = C >> 3, RY = 256 / CV;
  const int tx = threadIdx.x % CV, ty = threadIdx.x / CV;
  const int64_t stride = (int64_t)gridDim.x * RY;
  if (blockIdx.x == 0)                                   // the other set of accumulators: zero for the next BN call
    for (int i = threadIdx.x; i < zero_n; i += 256) acc_other[i] = 0.0;
  if (ty >= RY) return;
  float sc[8], sh[8], pv[8];
  { Raw8<T> p; p.ld(x + tx * 8); p.get(pv); }
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int c = tx * 8 + k;
    // plain (L1-cached) loads: every thread of the grid reads these 2 C doubles; through L2 alone (ld.cg) the few
    // cache lines they live in serialise the whole grid (measured: +15 us at 495 k rows)
    const double s1 = acc[c] * inv_n, s2 = acc[C + c] * inv_n;
    const double mean = (double)pv[k] + s1;
    double var = fma(-s1, s1, s2);
    if (var < 0.0) var = 0.0;
    const float m = (float)mean, is = inv_sqrt_refined(var + (double)eps);
    if (blockIdx.x == 0 && ty == 0) {
      const double unbiased = var * (double)n / (double)(n > 1 ? n - 1 : 1);
      running_mean[c] = (float)((double)momentum * running_mean[c] + (1.0 - (double)momentum) * mean);
      running_var[c] = (float)((double)momentum * running_var[c] + (1.0 - (double)momentum) * unbiased);
      save_mean[c] = m;
      save_invstd[c] = is;
    }
    sc[k] = is * (gamma ? gamma[c] : 1.f);
    sh[k] = (beta ? beta[c] : 0.f) - m * sc[k];
  }
  const T* px = x + tx * 8;
  T* po = out + tx * 8;
  int64_t r = (int64_t)blockIdx.x * RY + ty;
  for (; r + 3 * stride < n; r += 4 * stride) {
    Raw8<T> v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u].ld(px + (r + u * stride) * C);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float f[8];
      v[u].get(f);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float y = fmaf(f[k], sc[k], sh[k]);
        f[k] = (leak != 1.f && !(y > 0.f)) ? y * leak : y;
      }
      LoadVec<T, 8>::st(po + (r + u * stride) * C, f);
    }
  }
  for (; r < n; r += stride) {
    Raw8<T> v;
    v.ld(px + r * C);
    float f[8];
    v.get(f);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float y = fmaf(f[k], sc[k], sh[k]);
      f[k] = (leak != 1.f && !(y > 0.f)) ? y * leak : y;
    }
    LoadVec<T, 8>::st(po + r * C, f);
  }
}

template <typename T>
__global__ void __launch_bounds__(256, 3) k_bn_bwd_stats2(const T* __restrict__ x, const T* __restrict__ dout, int64_t n, int C,
                                                          const float* __restrict__ mean, const float* __restrict__ invstd,
                                                          const float* __restrict__ gamma, const float* __restrict__ beta,
                                                          float leak, double* acc) {
  __shared__ float sred[256 * 16];
  pdl_launch_dependents();
  pdl_wait();
  const int CV = C >> 3, RY = 256 / CV;
  const int tx = threadIdx.x % CV, ty = threadIdx.x / CV;
  const bool active = ty < RY;
  const int64_t stride = (int64_t)gridDim.x * RY;
  float a[8], b[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) a[k] = b[k] = 0.f;
  if (active) {
    // xhat = x * is + nm (nm = -mean * is); the fused leaky ReLU's mask is the sign of y = x * sc + sh, the very
    // expression the forward evaluated (sc = is * gamma, sh = beta - mean * sc)
    float is[8], nm[8], sc[8], sh[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = tx * 8 + k;
      is[k] = invstd[c];
      nm[k] = -mean[c] * is[k];
      sc[k] = is[k] * (gamma ? gamma[c] : 1.f);
      sh[k] = (beta ? beta[c] : 0.f) - mean[c] * sc[k];
    }
    const T* px = x + tx * 8;
    const T* pd = dout + tx * 8;
    auto body = [&](const Raw8<T>& rv, const Raw8<T>& rd) {
      float v[8], d[8];
      rv.get(v);
      rd.get(d);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float xh = fmaf(v[k], is[k], nm[k]);
        const float y = fmaf(v[k], sc[k], sh[k]);
        const float dd = (leak != 1.f && !(y > 0.f)) ? d[k] * leak : d[k];
        a[k] += dd;
        b[k] = fmaf(dd, xh, b[k]);
      }
    };
    int64_t r = (int64_t)blockIdx.x * RY + ty;
    for (; r + stride < n; r += 2 * stride) {
      Raw8<T> v[2], d[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) { v[u].ld(px + (r + u * stride) * C); d[u].ld(pd + (r + u * stride) * C); }
#pragma unroll
      for (int u = 0; u < 2; ++u) body(v[u], d[u]);
    }
    for (; r < n; r += stride) {
      Raw8<T> v, d;
      v.ld(px + r * C);
      d.ld(pd + r * C);
      body(v, d);
    }
  }
  block_col_sums<true>(a, b, C, CV, RY, tx, ty, active, sred, acc);
}

// COLSUM: also colsum[c] = sum over rows of the dx values as stored (colacc: C zeroed doubles, left zero)
template <typename T, bool COLSUM>
__global__ void __launch_bounds__(256, COLSUM ? 3 : 4) k_bn_bwd_apply2(const T* __restrict__ x, const T* __restrict__ dout, int64_t n, int C,
                                                          const float* __restrict__ mean, const float* __restrict__ invstd,
                                                          const float* __restrict__ gamma, const float* __restrict__ beta,
                                                          float leak, const double* __restrict__ acc,
                                                          double* __restrict__ acc_other, int zero_n, T* __restrict__ dx,
                                                          float* dgamma,
                                                          float* dbeta, int accumulate, double* colacc, unsigned* ticket,
                                                          float* __restrict__ colsum) {
  __shared__ float sred[COLSUM ? 256 * 8 : 1];
  pdl_launch_dependents();
  pdl_wait();
  const int CV = C >> 3, RY = 256 / CV;
  const int tx = threadIdx.x % CV, ty = threadIdx.x / CV;
  const bool active = ty < RY;
  const int64_t stride = (int64_t)gridDim.x * RY;
  if (blockIdx.x == 0)                                   // the other set of accumulators: zero for the next BN call
    for (int i = threadIdx.x; i < zero_n; i += 256) acc_other[i] = 0.0;
  float cs[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) cs[k] = 0.f;
  if (active) {
    // dx = gamma * is * (d - s1 - xhat * s2), xhat = (x - mean) * is, folded into three coefficients per channel:
    // dx = sc * d - (x * e2 + e1) with sc = gamma * is, e2 = sc * s2 * is, e1 = sc * (s1 - s2 * mean * is); the mask of
    // the fused leaky ReLU is the sign of y = x * sc + sh as in the forward
    float sc[8], sh[8], e1[8], e2[8];
    const float inv_n = n > 0 ? 1.f / (float)n : 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = tx * 8 + k;
      const double sa = acc[c], sb = acc[C + c];          // L1-cached on purpose (see k_bn_apply2)
      if (blockIdx.x == 0 && ty == 0) {
        if (dbeta) dbeta[c] = (accumulate ? dbeta[c] : 0.f) + (float)sa;
        if (dgamma) dgamma[c] = (accumulate ? dgamma[c] : 0.f) + (float)sb;
      }
      const float m = mean[c], is = invstd[c];
      sc[k] = is * (gamma ? gamma[c] : 1.f);
      sh[k] = (beta ? beta[c] : 0.f) - m * sc[k];
      const float s1 = (float)sa * inv_n, s2 = (float)sb * inv_n;
      e1[k] = sc[k] * (s1 - s2 * m * is);
      e2[k] = sc[k] * s2 * is;
    }
    const T* px = x + tx * 8;
    const T* pd = dout + tx * 8;
    T* po = dx + tx * 8;
    auto body = [&](const Raw8<T>& rv, const Raw8<T>& rd, T* dst) {
      float v[8], d[8];
      rv.get(v);
      rd.get(d);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float y = fmaf(v[k], sc[k], sh[k]);
        const float dd = (leak != 1.f && !(y > 0.f)) ? d[k] * leak : d[k];
        v[k] = fmaf(dd, sc[k], -fmaf(v[k], e2[k], e1[k]));
      }
      if (COLSUM) store8_sum(dst, v, cs);
      else LoadVec<T, 8>::st(dst, v);
    };
    int64_t r = (int64_t)blockIdx.x * RY + ty;
    for (; r + stride < n; r += 2 * stride) {
      Raw8<T> v[2], d[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) { v[u].ld(px + (r + u * stride) * C); d[u].ld(pd + (r + u * stride) * C); }
#pragma unroll
      for (int u = 0; u < 2; ++u) body(v[u], d[u], po + (r + u * stride) * C);
    }
    for (; r < n; r += stride) {
      Raw8<T> v, d;
      v.ld(px + r * C);
      d.ld(pd + r * C);
      body(v, d, po + r * C);
    }
  }
  if (COLSUM) {
    block_col_sums<false>(cs, nullptr, C, CV, RY, tx, ty, active, sred, colacc);
    if (!last_block(ticket)) return;
    for (int c = threadIdx.x; c < C; c += 256) {
      colsum[c] = (float)__ldcg(colacc + c);
      colacc[c] = 0.0;
    }
    if (threadIdx.x == 0) *ticket = 0u;
  }
}

// Column sums (conv bias gradient) in ONE launch: blocks add their partial sums to the zeroed fp64 accumulators, the
// last block to finish (atomic ticket) writes / accumulates the result and zeroes accumulators and ticket again.
// acc: [2048] doubles (zero on entry and exit), ticket: the unsigned right behind them.
template <typename T>
__global__ void __launch_bounds__(256) k_col_sum_fused(const T* __restrict__ x, int64_t n, int C, double* acc,
                                                       unsigned* ticket, float* __restrict__ out, int accumulate) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sred[];                        // [RY][CV][8]
  const int CV = C >> 3, RY = 256 / CV;
  const int tx = threadIdx.x % CV, ty = threadIdx.x / CV;
  float a[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) a[k] = 0.f;
  if (ty < RY) {
    for (int64_t r = (int64_t)blockIdx.x * RY + ty; r < n; r += (int64_t)gridDim.x * RY) {
      float v[8];
      LoadVec<T, 8>::ld(x + r * C + tx * 8, v);
#pragma unroll
      for (int k = 0; k < 8; ++k) a[k] += v[k];
    }
    float* dst = sred + ((size_t)ty * CV + tx) * 8;
#pragma unroll
    for (int k = 0; k < 8; ++k) dst[k] = a[k];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < CV * 8; i += 256) {
    float sum = 0.f;
    for (int y = 0; y < RY; ++y) sum += sred[((size_t)y * CV + (i >> 3)) * 8 + (i & 7)];
    atomicAdd(acc + i, (double)sum);
  }
  __threadfence();
  __syncthreads();
  __shared__ bool last;
  if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last) {
    __threadfence();
    for (int c = threadIdx.x; c < C; c += 256) {
      const double v = *reinterpret_cast<volatile double*>(acc + c);
      out[c] = (accumulate ? out[c] : 0.f) + (float)v;
      acc[c] = 0.0;
    }
    if (threadIdx.x == 0) *ticket = 0u;
  }
}

// fp64 accumulators of the two-launch BatchNorm kernels and k_col_sum_fused: 2 x 2048 doubles (BatchNorm) + 2048 doubles
// and a ticket (column sums) per (device, stream), allocated and zeroed once; every such kernel finds them zero and
// leaves them zero, so no memset precedes a launch.
constexpr int kAcc1 = 3 * 2048 + 2;          // second set of BatchNorm accumulators (2 x 2048 doubles) behind the tickets
constexpr size_t kScratchDoubles = (size_t)kAcc1 + 2 * 2048;
struct ScratchEntry { double* p = nullptr; unsigned phase = 0; int last_c[2] = {0, 0}; };
static std::mutex g_scratch_mu;
static std::map<std::pair<int, cudaStream_t>, ScratchEntry> g_scratch;
int zero_scratch(cudaStream_t s, double** out) {
  int dev = 0;
  SCN_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(g_scratch_mu);
  ScratchEntry& e = g_scratch[{dev, s}];
  if (e.p == nullptr) {
    double* p = nullptr;
    const cudaError_t err = cudaMalloc(&p, kScratchDoubles * sizeof(double));
    if (err != cudaSuccess) { (void)cudaGetLastError(); return (int)err; }
    const cudaError_t err2 = cudaMemsetAsync(p, 0, kScratchDoubles * sizeof(double), s);
    if (err2 != cudaSuccess) { cudaFree(p); return (int)err2; }
    e.p = p;
  }
  *out = e.p;
  return SCN_OK;
}
// which set of BatchNorm accumulators the next two-launch BatchNorm call of this stream uses (alternates per call)
// *zero_n: how many doubles of the OTHER set this call's apply kernel must clear -- what that set's last user (the
// previous call, possibly with more channels than this one) accumulated into
unsigned bn_next_phase(cudaStream_t s, int C, int* zero_n) {
  int dev = 0;
  (void)cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lock(g_scratch_mu);
  ScratchEntry& e = g_scratch[{dev, s}];
  const unsigned ph = e.phase & 1u;
  e.phase ^= 1u;
  *zero_n = 2 * e.last_c[ph ^ 1u];
  e.last_c[ph] = C;
  return ph;
}
// (Channel-sliced kernels -- one block per 8 channels over all rows, no grid barrier -- were measured for the small levels
// and are slower: 50 / 71 us against 36 / 24 us at 20 k rows x 160 channels: a warp then touches 32 different rows.)
// grid of the two-launch kernels: >= 4 rows per thread, at most one resident wave (per_sm blocks per SM)
int bn_grid2(int64_t n, int ry, int per_sm) {
  int64_t g = (n + (int64_t)ry * 4 - 1) / ((int64_t)ry * 4);
  const int64_t cap = (int64_t)kNumSMs * per_sm;
  if (g > cap) g = cap;
  return (int)(g < 1 ? 1 : g);
}

template <typename T, int VEC>
__global__ void k_bn_bwd_apply(const T* __restrict__ x, const T* __restrict__ dout, int64_t nvec, int C, int64_t n,
                               const float* __restrict__ mean, const float* __restrict__ invstd,
                               const float* __restrict__ gamma, const float* __restrict__ beta, float leak,
                               int training, const double* __restrict__ acc, T* __restrict__ dx) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= nvec) return;
  int c0 = (int)((i * VEC) % C);
  float v[VEC], d[VEC];
  LoadVec<T, VEC>::ld(x + i * VEC, v);
  LoadVec<T, VEC>::ld(dout + i * VEC, d);
  const float inv_n = n > 0 ? 1.f / (float)n : 0.f;
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    int c = c0 + k;
    float g = gamma ? gamma[c] : 1.f;
    float xh = (v[k] - mean[c]) * invstd[c];
    float y = xh * g + (beta ? beta[c] : 0.f);
    float dd = (leak != 1.f && !(y > 0.f)) ? d[k] * leak : d[k];
    float r = dd;
    if (training) r = dd - (float)acc[c] * inv_n - xh * (float)acc[C + c] * inv_n;
    v[k] = g * invstd[c] * r;
  }
  LoadVec<T, VEC>::st(dx + i * VEC, v);
}

__global__ void k_acc_to_float(const double* __restrict__ acc, int C, float* dgamma, float* dbeta, int accumulate) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  if (dbeta) dbeta[c] = (accumulate ? dbeta[c] : 0.f) + (float)acc[c];
  if (dgamma) dgamma[c] = (accumulate ? dgamma[c] : 0.f) + (float)acc[C + c];
}

template <typename T, int VEC>
__global__ void k_leaky_fwd(const T* __restrict__ x, int64_t nvec, float leak, T* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= nvec) return;
  float v[VEC];
  LoadVec<T, VEC>::ld(x + i * VEC, v);
#pragma unroll
  for (int k = 0; k < VEC; ++k) v[k] = v[k] > 0.f ? v[k] : v[k] * leak;
  LoadVec<T, VEC>::st(out + i * VEC, v);
}
template <typename T, int VEC>
__global__ void k_leaky_bwd(const T* __restrict__ x, const T* __restrict__ dout, int64_t nvec, float leak,
                            T* __restrict__ dx) {
  pdl_launch_dependents();
  pdl_wait();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= nvec) return;
  float v[VEC], d[VEC];
  LoadVec<T, VEC>::ld(x + i * VEC, v);
  LoadVec<T, VEC>::ld(dout + i * VEC, d);
#pragma unroll
  for (int k = 0; k < VEC; ++k) d[k] = v[k] > 0.f ? d[k] : d[k] * leak;
  LoadVec<T, VEC>::st(dx + i * VEC, d);
}
template <typename T, int VEC>
__global__ void k_add_fwd(const T* __restrict__ a, const T* __restrict__ b, int64_t nvec, float leak,
                          T* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= nvec) return;
  float v[VEC], w[VEC];
  LoadVec<T, VEC>::ld(a + i * VEC, v);
  LoadVec<T, VEC>::ld(b + i * VEC, w);
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    float s = v[k] + w[k];
    v[k] = (leak != 1.f && !(s > 0.f)) ? s * leak : s;
  }
  LoadVec<T, VEC>::st(out + i * VEC, v);
}

__global__ void k_input_scatter(const float* __restrict__ in, const int32_t* __restrict__ rows, int64_t n_in, int C,
                                float* __restrict__ out, float* __restrict__ cnt) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_in * C) return;
  int64_t r = i / C;
  int c = (int)(i - r * C);
  atomicAdd(out + (int64_t)rows[r] * C + c, in[i]);
  if (cnt && c == 0) atomicAdd(cnt + rows[r], 1.f);
}
__global__ void k_div_rows(float* __restrict__ out, const float* __restrict__ cnt, int64_t n, int C) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n * C) return;
  out[i] /= cnt[i / C];
}
template <typename TI, typename TO>
__global__ void k_convert(const TI* __restrict__ in, int64_t n, TO* __restrict__ out) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) Elem<TO>::st(out + i, Elem<TI>::ld(in + i));
}
template <typename TI, typename TO>
__global__ void k_rows_gather(const TI* __restrict__ src, const int32_t* __restrict__ rows, int64_t n_rows, int C,
                              TO* __restrict__ out) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_rows * C) return;
  int64_t r = i / C;
  int c = (int)(i - r * C);
  Elem<TO>::st(out + i, Elem<TI>::ld(src + (int64_t)rows[r] * C + c));
}
template <typename TI>
__global__ void k_rows_scatter_add(const TI* __restrict__ src, const int32_t* __restrict__ rows, int64_t n_rows, int C,
                                   float* __restrict__ out) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_rows * C) return;
  int64_t r = i / C;
  int c = (int)(i - r * C);
  atomicAdd(out + (int64_t)rows[r] * C + c, Elem<TI>::ld(src + i));
}

// AveragePooling rows: out[r, :] = scale * sum_k x[nbr[k][r], :] over the table entries that exist (k ascending, fp32
// accumulation: deterministic).  The same kernel is the backward with the transposed table.  ldx = source row stride
// in elements (nFeaturesToDrop reads a column window of a wider matrix).
template <typename T, int V>
__global__ void k_pool_rows(const T* __restrict__ x, int ldx, const int32_t* __restrict__ nbr, int K, int64_t n_rows,
                            int64_t n_pad, int C, float scale, T* __restrict__ out) {
  const int cg = C / V;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_rows * cg) return;
  int64_t r = i / cg;
  int c = (int)(i - r * cg) * V;
  float acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = 0.f;
  for (int k = 0; k < K; ++k) {
    int32_t s = __ldg(nbr + (int64_t)k * n_pad + r);
    if (s < 0) continue;
    const T* src = x + (int64_t)s * ldx + c;
    if constexpr (V == 4) {
      float4 t = ld4(src);
      acc[0] += t.x; acc[1] += t.y; acc[2] += t.z; acc[3] += t.w;
    } else {
      acc[0] += Elem<T>::ld(src);
    }
  }
  T* dst = out + r * C + c;
  if constexpr (V == 4) st4(dst, make_float4(acc[0] * scale, acc[1] * scale, acc[2] * scale, acc[3] * scale));
  else Elem<T>::st(dst, acc[0] * scale);
}

template <typename T>
__global__ void k_s2d_fwd(const T* __restrict__ x, const uint64_t* __restrict__ keys, int64_t n, int C, int batch, int s0,
                          int s1, int s2, float* __restrict__ dense) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n * C) return;
  int64_t r = i / C;
  int c = (int)(i - r * C);
  int x0, x1, x2, b;
  key_unpack(keys[r], x0, x1, x2, b);
  if (x0 >= s0 || x1 >= s1 || x2 >= s2 || b >= batch) return;      // a site outside the dense volume is dropped, never written
  dense[((((int64_t)b * C + c) * s0 + x0) * s1 + x1) * s2 + x2] = Elem<T>::ld(x + i);
}
template <typename T>
__global__ void k_s2d_bwd(const float* __restrict__ ddense, const uint64_t* __restrict__ keys, int64_t n, int C, int batch,
                          int s0, int s1, int s2, T* __restrict__ dx) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n * C) return;
  int64_t r = i / C;
  int c = (int)(i - r * C);
  int x0, x1, x2, b;
  key_unpack(keys[r], x0, x1, x2, b);
  float v = 0.f;
  if (x0 < s0 && x1 < s1 && x2 < s2 && b < batch) v = ddense[((((int64_t)b * C + c) * s0 + x0) * s1 + x1) * s2 + x2];
  Elem<T>::st(dx + i, v);
}

// What the last call of each launcher below launched (developer entry like scn_tc_debug_last_launch, for the tests'
// coverage check), written on the host before the launches.  Records: BatchNorm forward, BatchNorm backward, column
// sum, LeakyReLU / AddTable, AveragePooling; fields:
//   path    BatchNorm: 2 two-launch, 4 four-launch; column sum: 1 k_col_sum_fused, 4 k_col_reduce2;
//           LeakyReLU / AddTable: 0 leaky forward, 1 leaky backward, 2 add
//   vec     VEC of the statistics / column reduction (0: none, eval-mode forward), or of the elementwise / pool kernel
//   apply   BatchNorm apply form: 1 row-streaming, 2 element-indexed
//   avec    VEC of the apply kernel
//   grid    grid of the statistics / reduction kernel (x), or of the elementwise / pool kernel
//   grid2   grid of the apply kernel
//   slices  k_col_reduce2's channel slices (gridDim.y)
//   colsum  BatchNorm backward: 0 no column sums of dx, 1 fused into the apply kernel, 2 a separate column-sum call
enum { kEwBnFwd = 0, kEwBnBwd = 1, kEwColSum = 2, kEwElem = 3, kEwPool = 4, kEwRecords = 5, kEwFields = 8 };
static int32_t g_ew_last_launch[kEwRecords][kEwFields] = {};
void ew_record(int which, int path, int vec, int apply, int avec, int64_t grid, int64_t grid2, int slices, int colsum) {
  const int32_t rec[kEwFields] = {path, vec, apply, avec, (int32_t)grid, (int32_t)grid2, slices, colsum};
  for (int i = 0; i < kEwFields; ++i) g_ew_last_launch[which][i] = rec[i];
}

// rec: the launch record whose reduction fields (vec, grid, slices) this launch fills in
template <int VEC, typename F>
int launch_col_reduce(F f, int64_t n, int C, double* acc, cudaStream_t s, int32_t* rec) {
  const int groups = C / VEC;
  const int slices = (groups + kRedThreads - 1) / kRedThreads;
  const int CV = (groups + slices - 1) / slices;        // <= 256 channel groups per block, slices as even as possible
  const int RY = kRedThreads / CV;
  const size_t smem = (size_t)RY * CV * 2 * VEC * sizeof(float);
  const unsigned g = (unsigned)((n + kRedRows - 1) / kRedRows);
  rec[1] = VEC; rec[4] = (int32_t)g; rec[6] = slices;
  k_col_reduce2<VEC, F><<<dim3(g, (unsigned)slices), kRedThreads, smem, s>>>(f, n, C, CV, acc);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

template <typename T>
int bn_forward_t(const T* x, int64_t n, int C, const float* gamma, const float* beta, float* rm, float* rv,
                 int training, float eps, float momentum, float leak, float* save_mean, float* save_invstd,
                 double* ws, T* out, cudaStream_t s) {
  const bool vec = (C % 4) == 0 && (((uintptr_t)x | (uintptr_t)out) % (4 * sizeof(T))) == 0;
  const bool vec8 = (C % 8) == 0 && (((uintptr_t)x | (uintptr_t)out) & 15) == 0;
  int32_t* rec = g_ew_last_launch[kEwBnFwd];
  if (training && vec8 && C <= 2048 && n > 0) {
    double* zws = nullptr;
    const int rc = zero_scratch(s, &zws);
    if (rc != SCN_OK) return rc;
    const int ry = 256 / (C >> 3);
    const int g = bn_grid2(n, ry, 4);
    int zero_n = 0;
    const unsigned ph = bn_next_phase(s, C, &zero_n);
    double* acc = zws + (ph ? kAcc1 : 0);
    double* other = zws + (ph ? 0 : kAcc1);
    ew_record(kEwBnFwd, 2, 8, 1, 8, g, g, 0, 0);
    SCN_CUDA(scn_launch_pdl(k_bn_stats2<T>, dim3((unsigned)g), dim3(256), 0, s, x, n, C, acc));
    SCN_LAUNCH_CHECK();
    SCN_CUDA(scn_launch_pdl(k_bn_apply2<T>, dim3((unsigned)g), dim3(256), 0, s, x, n, C, gamma, beta, rm, rv, eps, momentum, leak,
                            save_mean, save_invstd, (const double*)acc, other, zero_n, 1.0 / (double)n, out));
    SCN_LAUNCH_CHECK();
    return SCN_OK;
  }
  ew_record(kEwBnFwd, 4, 0, 0, 0, 0, 0, 0, 0);
  if (training) {
    SCN_CUDA(cudaMemsetAsync(ws, 0, 2 * (size_t)C * sizeof(double), s));
    if (n > 0) {
      int rc = vec8 ? launch_col_reduce<8>(StatsF<T, 8>{x, C}, n, C, ws, s, rec)
               : vec ? launch_col_reduce<4>(StatsF<T, 4>{x, C}, n, C, ws, s, rec)
                     : launch_col_reduce<1>(StatsF<T, 1>{x, C}, n, C, ws, s, rec);
      if (rc) return rc;
    }
  }
  k_bn_finalize<T><<<grid_for(C, 128), 128, 0, s>>>(ws, x, n, C, training, eps, momentum, rm, rv, save_mean,
                                                    save_invstd);
  SCN_LAUNCH_CHECK();
  if (n == 0) return SCN_OK;
  int64_t total = n * C;
  if (vec8 && C <= 2048) {
    const int ry = 256 / (C >> 3);
    int64_t g = (n + (int64_t)ry * 4 - 1) / ((int64_t)ry * 4);      // >= 4 rows per thread
    if (g > (int64_t)kNumSMs * 8) g = (int64_t)kNumSMs * 8;
    if (g < 1) g = 1;
    rec[2] = 1; rec[3] = 8; rec[5] = (int32_t)g;
    k_bn_apply_rows<T><<<(unsigned)g, 256, 0, s>>>(x, n, C, save_mean, save_invstd, gamma, beta, leak, out);
  } else if (vec) {
    rec[2] = 2; rec[3] = 4; rec[5] = (int32_t)grid_for(total / 4, 256);
    k_bn_apply<T, 4><<<grid_for(total / 4, 256), 256, 0, s>>>(x, total / 4, C, save_mean, save_invstd, gamma, beta,
                                                              leak, out);
  } else {
    rec[2] = 2; rec[3] = 1; rec[5] = (int32_t)grid_for(total, 256);
    k_bn_apply<T, 1><<<grid_for(total, 256), 256, 0, s>>>(x, total, C, save_mean, save_invstd, gamma, beta, leak, out);
  }
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

template <typename T>
int bn_backward_t(const T* x, const T* dout, int64_t n, int C, const float* gamma, const float* beta,
                  const float* mean, const float* invstd, int training, float leak, double* ws, T* dx,
                  float* dgamma, float* dbeta, int accumulate, float* colsum, cudaStream_t s) {
  const bool vec = (C % 4) == 0 && (((uintptr_t)x | (uintptr_t)dout | (uintptr_t)dx) % (4 * sizeof(T))) == 0;
  const bool vec8 = (C % 8) == 0 && (((uintptr_t)x | (uintptr_t)dout | (uintptr_t)dx) & 15) == 0;
  int32_t* rec = g_ew_last_launch[kEwBnBwd];
  if (training && vec8 && C <= 2048 && n > 0) {
    double* zws = nullptr;
    const int rc = zero_scratch(s, &zws);
    if (rc != SCN_OK) return rc;
    const int ry = 256 / (C >> 3);
    int zero_n = 0;
    const unsigned ph = bn_next_phase(s, C, &zero_n);
    double* acc = zws + (ph ? kAcc1 : 0);
    double* other = zws + (ph ? 0 : kAcc1);
    double* colacc = zws + 2 * 2048;                                   // shared with k_col_sum_fused (stream-ordered)
    unsigned* ticket = reinterpret_cast<unsigned*>(zws + 3 * 2048 + 1);
    ew_record(kEwBnBwd, 2, 8, 1, 8, bn_grid2(n, ry, 3), bn_grid2(n, ry, colsum ? 3 : 4), 0, colsum ? 1 : 0);
    SCN_CUDA(scn_launch_pdl(k_bn_bwd_stats2<T>, dim3((unsigned)bn_grid2(n, ry, 3)), dim3(256), 0, s, x, dout, n, C, mean, invstd,
                            gamma, beta, leak, acc));
    SCN_LAUNCH_CHECK();
    if (colsum)
      SCN_CUDA(scn_launch_pdl(k_bn_bwd_apply2<T, true>, dim3((unsigned)bn_grid2(n, ry, 3)), dim3(256), 0, s, x, dout, n, C, mean,
                              invstd, gamma, beta, leak, (const double*)acc, other, zero_n, dx, dgamma, dbeta, accumulate,
                              colacc, ticket, colsum));
    else
      SCN_CUDA(scn_launch_pdl(k_bn_bwd_apply2<T, false>, dim3((unsigned)bn_grid2(n, ry, 4)), dim3(256), 0, s, x, dout, n, C, mean,
                              invstd, gamma, beta, leak, (const double*)acc, other, zero_n, dx, dgamma, dbeta, accumulate,
                              colacc, ticket, (float*)nullptr));
    SCN_LAUNCH_CHECK();
    return SCN_OK;
  }
  ew_record(kEwBnBwd, 4, 0, 0, 0, 0, 0, 0, colsum ? 2 : 0);
  SCN_CUDA(cudaMemsetAsync(ws, 0, 2 * (size_t)C * sizeof(double), s));
  if (n > 0) {
    int rc = vec8 ? launch_col_reduce<8>(BnBwdF<T, 8>{x, dout, mean, invstd, gamma, beta, leak, C}, n, C, ws, s, rec)
             : vec ? launch_col_reduce<4>(BnBwdF<T, 4>{x, dout, mean, invstd, gamma, beta, leak, C}, n, C, ws, s, rec)
                   : launch_col_reduce<1>(BnBwdF<T, 1>{x, dout, mean, invstd, gamma, beta, leak, C}, n, C, ws, s, rec);
    if (rc) return rc;
  }
  k_acc_to_float<<<grid_for(C, 128), 128, 0, s>>>(ws, C, dgamma, dbeta, accumulate);
  SCN_LAUNCH_CHECK();
  if (n == 0) {
    if (colsum) SCN_CUDA(cudaMemsetAsync(colsum, 0, (size_t)C * sizeof(float), s));
    return SCN_OK;
  }
  int64_t total = n * C;
  if (vec8 && C <= 2048) {
    const int ry = 256 / (C >> 3);
    int64_t g = (n + (int64_t)ry * 4 - 1) / ((int64_t)ry * 4);
    if (g > (int64_t)kNumSMs * 8) g = (int64_t)kNumSMs * 8;
    if (g < 1) g = 1;
    rec[2] = 1; rec[3] = 8; rec[5] = (int32_t)g;
    k_bn_bwd_apply_rows<T><<<(unsigned)g, 256, 0, s>>>(x, dout, n, C, mean, invstd, gamma, beta, leak, training, ws, dx);
  } else if (vec) {
    rec[2] = 2; rec[3] = 4; rec[5] = (int32_t)grid_for(total / 4, 256);
    k_bn_bwd_apply<T, 4><<<grid_for(total / 4, 256), 256, 0, s>>>(x, dout, total / 4, C, n, mean, invstd, gamma, beta,
                                                                  leak, training, ws, dx);
  } else {
    rec[2] = 2; rec[3] = 1; rec[5] = (int32_t)grid_for(total, 256);
    k_bn_bwd_apply<T, 1><<<grid_for(total, 256), 256, 0, s>>>(x, dout, total, C, n, mean, invstd, gamma, beta, leak,
                                                              training, ws, dx);
  }
  SCN_LAUNCH_CHECK();
  if (colsum)      // paths without the fused column sums: one more pass over dx
    return scn_col_sum(dx, std::is_same<T, float>::value ? SCN_F32 : SCN_BF16, n, C, ws, colsum, s);
  return SCN_OK;
}

#define DISPATCH_T(dtype, CALL_F32, CALL_BF16)          \
  switch (dtype) {                                      \
    case SCN_F32: { CALL_F32; break; }                  \
    case SCN_BF16: { CALL_BF16; break; }                \
    default: return SCN_ERR_ARG;                        \
  }

template <typename T>
int ew_launch3(int which, const T* a, const T* b, int64_t count, float leak, T* out, cudaStream_t s) {
  if (count == 0) return SCN_OK;
  bool vec = (count % 4 == 0) && ((((uintptr_t)a | (uintptr_t)b | (uintptr_t)out) & 15) == 0);
  if (vec && count % 8 == 0) {                 // 16-byte accesses for bf16, 2 x 16 bytes for fp32
    const int64_t n8 = count / 8;
    const unsigned g8 = grid_for(n8, 256);
    ew_record(kEwElem, which, 8, 0, 0, g8, 0, 0, 0);
    if (which == 0) SCN_CUDA(scn_launch_pdl(k_leaky_fwd<T, 8>, dim3(g8), dim3(256), 0, s, a, n8, leak, out));
    else if (which == 1) SCN_CUDA(scn_launch_pdl(k_leaky_bwd<T, 8>, dim3(g8), dim3(256), 0, s, a, b, n8, leak, out));
    else SCN_CUDA(scn_launch_pdl(k_add_fwd<T, 8>, dim3(g8), dim3(256), 0, s, a, b, n8, leak, out));
    SCN_LAUNCH_CHECK();
    return SCN_OK;
  }
  int64_t nv = vec ? count / 4 : count;
  unsigned g = grid_for(nv, 256);
  ew_record(kEwElem, which, vec ? 4 : 1, 0, 0, g, 0, 0, 0);
  if (which == 0) {
    if (vec) k_leaky_fwd<T, 4><<<g, 256, 0, s>>>(a, nv, leak, out); else k_leaky_fwd<T, 1><<<g, 256, 0, s>>>(a, nv, leak, out);
  } else if (which == 1) {
    if (vec) k_leaky_bwd<T, 4><<<g, 256, 0, s>>>(a, b, nv, leak, out); else k_leaky_bwd<T, 1><<<g, 256, 0, s>>>(a, b, nv, leak, out);
  } else {
    if (vec) k_add_fwd<T, 4><<<g, 256, 0, s>>>(a, b, nv, leak, out); else k_add_fwd<T, 1><<<g, 256, 0, s>>>(a, b, nv, leak, out);
  }
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

}  // namespace

extern "C" void scn_ew_debug_last_launch(int32_t* out) {
  for (int r = 0; r < kEwRecords; ++r)
    for (int i = 0; i < kEwFields; ++i) out[r * kEwFields + i] = g_ew_last_launch[r][i];
}

extern "C" int scn_bn_forward(const void* x, int dtype, int64_t n, int C, const float* gamma, const float* beta,
                              float* running_mean, float* running_var, int training, float eps, float momentum,
                              float leakiness, float* save_mean, float* save_invstd, double* stats_ws, void* out,
                              void* stream) {
  if (C < 1 || !running_mean || !running_var || !save_mean || !save_invstd || !stats_ws) return SCN_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  DISPATCH_T(dtype,
             return bn_forward_t<float>((const float*)x, n, C, gamma, beta, running_mean, running_var, training, eps,
                                        momentum, leakiness, save_mean, save_invstd, stats_ws, (float*)out, s),
             return bn_forward_t<__nv_bfloat16>((const __nv_bfloat16*)x, n, C, gamma, beta, running_mean, running_var,
                                                training, eps, momentum, leakiness, save_mean, save_invstd, stats_ws,
                                                (__nv_bfloat16*)out, s));
  return SCN_OK;
}

extern "C" int scn_bn_backward_colsum(const void* x, const void* dout, int dtype, int64_t n, int C, const float* gamma,
                                      const float* beta, const float* save_mean, const float* save_invstd, int training,
                                      float leakiness, double* stats_ws, void* dx, float* dgamma, float* dbeta,
                                      int accumulate_params, float* dx_colsum, void* stream) {
  if (C < 1 || !save_mean || !save_invstd || !stats_ws) return SCN_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  DISPATCH_T(dtype,
             return bn_backward_t<float>((const float*)x, (const float*)dout, n, C, gamma, beta, save_mean, save_invstd,
                                         training, leakiness, stats_ws, (float*)dx, dgamma, dbeta, accumulate_params,
                                         dx_colsum, s),
             return bn_backward_t<__nv_bfloat16>((const __nv_bfloat16*)x, (const __nv_bfloat16*)dout, n, C, gamma, beta,
                                                 save_mean, save_invstd, training, leakiness, stats_ws,
                                                 (__nv_bfloat16*)dx, dgamma, dbeta, accumulate_params, dx_colsum, s));
  return SCN_OK;
}

extern "C" int scn_bn_backward(const void* x, const void* dout, int dtype, int64_t n, int C, const float* gamma,
                               const float* beta, const float* save_mean, const float* save_invstd, int training,
                               float leakiness, double* stats_ws, void* dx, float* dgamma, float* dbeta,
                               int accumulate_params, void* stream) {
  return scn_bn_backward_colsum(x, dout, dtype, n, C, gamma, beta, save_mean, save_invstd, training, leakiness, stats_ws,
                                dx, dgamma, dbeta, accumulate_params, nullptr, stream);
}

extern "C" int scn_col_sum(const void* x, int dtype, int64_t n, int C, double* stats_ws, float* out, void* stream) {
  return scn_col_sum_acc(x, dtype, n, C, stats_ws, out, 0, stream);
}

extern "C" int scn_col_sum_acc(const void* x, int dtype, int64_t n, int C, double* stats_ws, float* out, int accumulate,
                               void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (C < 1 || !out || !stats_ws) return SCN_ERR_ARG;
  if (n > 0 && (C % 8) == 0 && C <= 2048 && (((uintptr_t)x) & 15) == 0) {
    double* z = nullptr;
    const int rc = zero_scratch(s, &z);
    if (rc != SCN_OK) return rc;
    double* acc1 = z + 2 * 2048;
    unsigned* ticket = reinterpret_cast<unsigned*>(z + 3 * 2048);
    const int ry = 256 / (C >> 3);
    int64_t g = (n + (int64_t)ry * 8 - 1) / ((int64_t)ry * 8);
    if (g > (int64_t)kNumSMs * 4) g = (int64_t)kNumSMs * 4;
    if (g < 1) g = 1;
    const size_t smem = (size_t)ry * (C >> 3) * 8 * sizeof(float);
    ew_record(kEwColSum, 1, 8, 0, 0, g, 0, 0, 0);
    if (dtype == SCN_F32)
      SCN_CUDA(scn_launch_pdl(k_col_sum_fused<float>, dim3((unsigned)g), dim3(256), smem, s, (const float*)x, n, C, acc1, ticket, out, accumulate));
    else if (dtype == SCN_BF16)
      SCN_CUDA(scn_launch_pdl(k_col_sum_fused<__nv_bfloat16>, dim3((unsigned)g), dim3(256), smem, s, (const __nv_bfloat16*)x, n, C, acc1,
                              ticket, out, accumulate));
    else
      return SCN_ERR_ARG;
    SCN_LAUNCH_CHECK();
    return SCN_OK;
  }
  double* acc = stats_ws;
  ew_record(kEwColSum, 4, 0, 0, 0, 0, 0, 0, 0);
  int32_t* rec = g_ew_last_launch[kEwColSum];
  SCN_CUDA(cudaMemsetAsync(acc, 0, 2 * (size_t)C * sizeof(double), s));
  int rc = SCN_OK;
  if (n > 0) {
    const size_t esz = dtype == SCN_F32 ? sizeof(float) : sizeof(__nv_bfloat16);
    const bool vec = (C % 4) == 0 && ((uintptr_t)x % (4 * esz)) == 0;
    if (dtype == SCN_F32)
      rc = vec ? launch_col_reduce<4>(SumF<float, 4>{(const float*)x, C}, n, C, acc, s, rec)
               : launch_col_reduce<1>(SumF<float, 1>{(const float*)x, C}, n, C, acc, s, rec);
    else if (dtype == SCN_BF16)
      rc = vec ? launch_col_reduce<4>(SumF<__nv_bfloat16, 4>{(const __nv_bfloat16*)x, C}, n, C, acc, s, rec)
               : launch_col_reduce<1>(SumF<__nv_bfloat16, 1>{(const __nv_bfloat16*)x, C}, n, C, acc, s, rec);
    else
      rc = SCN_ERR_ARG;
  }
  if (rc != SCN_OK) return rc;
  k_acc_to_float<<<grid_for(C, 128), 128, 0, s>>>(acc, C, nullptr, out, accumulate);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

extern "C" int scn_leaky_forward(const void* x, int dtype, int64_t count, float leak, void* out, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  DISPATCH_T(dtype, return ew_launch3<float>(0, (const float*)x, nullptr, count, leak, (float*)out, s),
             return ew_launch3<__nv_bfloat16>(0, (const __nv_bfloat16*)x, nullptr, count, leak, (__nv_bfloat16*)out, s));
  return SCN_OK;
}
extern "C" int scn_leaky_backward(const void* x, const void* dout, int dtype, int64_t count, float leak, void* dx,
                                  void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  DISPATCH_T(dtype, return ew_launch3<float>(1, (const float*)x, (const float*)dout, count, leak, (float*)dx, s),
             return ew_launch3<__nv_bfloat16>(1, (const __nv_bfloat16*)x, (const __nv_bfloat16*)dout, count, leak,
                                              (__nv_bfloat16*)dx, s));
  return SCN_OK;
}
extern "C" int scn_add_forward(const void* a, const void* b, int dtype, int64_t count, float leak, void* out,
                               void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  DISPATCH_T(dtype, return ew_launch3<float>(2, (const float*)a, (const float*)b, count, leak, (float*)out, s),
             return ew_launch3<__nv_bfloat16>(2, (const __nv_bfloat16*)a, (const __nv_bfloat16*)b, count, leak,
                                              (__nv_bfloat16*)out, s));
  return SCN_OK;
}

extern "C" int scn_input_layer_forward(const float* in, const int32_t* row_of_input, int64_t n_in, int64_t n_active,
                                       int C, int mode, void* out, int out_dtype, float* count_ws, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (mode == 1 || mode == 2) return SCN_ERR_UNSUPPORTED;   // last/first-wins: not used by the reference
  if (out_dtype != SCN_F32) return SCN_ERR_UNSUPPORTED;     // accumulate in fp32; cast afterwards
  if (n_active == 0) return SCN_OK;
  if (!out || !in || !row_of_input) return SCN_ERR_ARG;
  SCN_CUDA(cudaMemsetAsync(out, 0, (size_t)n_active * C * sizeof(float), s));
  float* cnt = nullptr;
  if (mode == 4) {
    if (!count_ws) return SCN_ERR_WORKSPACE;
    cnt = count_ws;
    SCN_CUDA(cudaMemsetAsync(cnt, 0, (size_t)n_active * sizeof(float), s));
  }
  k_input_scatter<<<grid_for(n_in * C, 256), 256, 0, s>>>(in, row_of_input, n_in, C, (float*)out, cnt);
  SCN_LAUNCH_CHECK();
  if (mode == 4) {
    k_div_rows<<<grid_for(n_active * C, 256), 256, 0, s>>>((float*)out, cnt, n_active, C);
    SCN_LAUNCH_CHECK();
  }
  return SCN_OK;
}

extern "C" int scn_rows_gather(const void* src, int dtype, const int32_t* rows, int64_t n_rows, int C, void* out,
                               int out_dtype, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n_rows == 0) return SCN_OK;
  unsigned g = grid_for(n_rows * C, 256);
  if (rows == nullptr) {   // plain dtype conversion of a [n_rows, C] matrix
    int64_t n = n_rows * C;
    if (dtype == SCN_F32 && out_dtype == SCN_BF16) k_convert<float, __nv_bfloat16><<<g, 256, 0, s>>>((const float*)src, n, (__nv_bfloat16*)out);
    else if (dtype == SCN_BF16 && out_dtype == SCN_F32) k_convert<__nv_bfloat16, float><<<g, 256, 0, s>>>((const __nv_bfloat16*)src, n, (float*)out);
    else if (dtype == SCN_F32 && out_dtype == SCN_F32) k_convert<float, float><<<g, 256, 0, s>>>((const float*)src, n, (float*)out);
    else if (dtype == SCN_BF16 && out_dtype == SCN_BF16) k_convert<__nv_bfloat16, __nv_bfloat16><<<g, 256, 0, s>>>((const __nv_bfloat16*)src, n, (__nv_bfloat16*)out);
    else return SCN_ERR_ARG;
    SCN_LAUNCH_CHECK();
    return SCN_OK;
  }
  if (dtype == SCN_F32 && out_dtype == SCN_F32) k_rows_gather<float, float><<<g, 256, 0, s>>>((const float*)src, rows, n_rows, C, (float*)out);
  else if (dtype == SCN_F32 && out_dtype == SCN_BF16) k_rows_gather<float, __nv_bfloat16><<<g, 256, 0, s>>>((const float*)src, rows, n_rows, C, (__nv_bfloat16*)out);
  else if (dtype == SCN_BF16 && out_dtype == SCN_F32) k_rows_gather<__nv_bfloat16, float><<<g, 256, 0, s>>>((const __nv_bfloat16*)src, rows, n_rows, C, (float*)out);
  else if (dtype == SCN_BF16 && out_dtype == SCN_BF16) k_rows_gather<__nv_bfloat16, __nv_bfloat16><<<g, 256, 0, s>>>((const __nv_bfloat16*)src, rows, n_rows, C, (__nv_bfloat16*)out);
  else return SCN_ERR_ARG;
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

extern "C" int scn_rows_scatter_add(const void* src, int dtype, const int32_t* rows, int64_t n_rows, int C,
                                    float* out_f32, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n_rows == 0) return SCN_OK;
  if (!src || !rows || !out_f32) return SCN_ERR_ARG;
  unsigned g = grid_for(n_rows * C, 256);
  if (dtype == SCN_F32) k_rows_scatter_add<float><<<g, 256, 0, s>>>((const float*)src, rows, n_rows, C, out_f32);
  else if (dtype == SCN_BF16) k_rows_scatter_add<__nv_bfloat16><<<g, 256, 0, s>>>((const __nv_bfloat16*)src, rows, n_rows, C, out_f32);
  else return SCN_ERR_ARG;
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

template <typename T>
static int launch_pool_rows(const void* x, int ldx, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int C,
                            float scale, void* out, cudaStream_t s) {
  const size_t vb = 4 * sizeof(T);      // bytes of one 4-element access
  const bool vec = C % 4 == 0 && ldx % 4 == 0 && (uintptr_t)x % vb == 0 && (uintptr_t)out % vb == 0;
  ew_record(kEwPool, 0, vec ? 4 : 1, 0, 0, vec ? grid_for(n_rows * (C / 4), 256) : grid_for(n_rows * C, 256), 0, 0, 0);
  if (vec)
    k_pool_rows<T, 4><<<grid_for(n_rows * (C / 4), 256), 256, 0, s>>>((const T*)x, ldx, nbr, K, n_rows, n_pad, C, scale,
                                                                       (T*)out);
  else
    k_pool_rows<T, 1><<<grid_for(n_rows * C, 256), 256, 0, s>>>((const T*)x, ldx, nbr, K, n_rows, n_pad, C, scale,
                                                                 (T*)out);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

extern "C" int scn_pool_rows(const void* x, int dtype, int ldx, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad,
                             int C, float scale, void* out, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n_rows == 0 || C == 0) return SCN_OK;
  if (!x || !nbr || !out || K < 1 || C < 0 || ldx < C || n_pad < n_rows) return SCN_ERR_ARG;
  if (dtype == SCN_F32) return launch_pool_rows<float>(x, ldx, nbr, K, n_rows, n_pad, C, scale, out, s);
  if (dtype == SCN_BF16) return launch_pool_rows<__nv_bfloat16>(x, ldx, nbr, K, n_rows, n_pad, C, scale, out, s);
  return SCN_ERR_ARG;
}

extern "C" int scn_sparse_to_dense_forward(const void* x, int dtype, const uint64_t* keys, int64_t n, int C, int batch,
                                           int s0, int s1, int s2, float* dense, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  size_t total = (size_t)batch * C * s0 * s1 * s2;
  if (total == 0) return SCN_OK;
  if (!dense) return SCN_ERR_ARG;
  SCN_CUDA(cudaMemsetAsync(dense, 0, total * sizeof(float), s));
  if (n == 0) return SCN_OK;
  unsigned g = grid_for(n * C, 256);
  if (dtype == SCN_F32) k_s2d_fwd<float><<<g, 256, 0, s>>>((const float*)x, keys, n, C, batch, s0, s1, s2, dense);
  else if (dtype == SCN_BF16) k_s2d_fwd<__nv_bfloat16><<<g, 256, 0, s>>>((const __nv_bfloat16*)x, keys, n, C, batch, s0, s1, s2, dense);
  else return SCN_ERR_ARG;
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

extern "C" int scn_sparse_to_dense_backward(const float* ddense, const uint64_t* keys, int64_t n, int C, int batch,
                                            int s0, int s1, int s2, void* dx, int dtype, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n == 0) return SCN_OK;
  unsigned g = grid_for(n * C, 256);
  if (dtype == SCN_F32) k_s2d_bwd<float><<<g, 256, 0, s>>>(ddense, keys, n, C, batch, s0, s1, s2, (float*)dx);
  else if (dtype == SCN_BF16) k_s2d_bwd<__nv_bfloat16><<<g, 256, 0, s>>>(ddense, keys, n, C, batch, s0, s1, s2, (__nv_bfloat16*)dx);
  else return SCN_ERR_ARG;
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}
