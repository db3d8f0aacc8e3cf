// Convolution arithmetic, first generation: output-stationary gather-GEMM on the neighbour table.
//   * exact fp32 FMA kernels (precision SCN_PREC_FP32, odd channel counts, and the Cin=1 stem in that mode)
//   * bf16-operand / fp32-accumulate tensor-core kernels built on mma.sync (HMMA): the fp32 features of the "mixed"
//     mode, and the bf16 weight gradient where the tcgen05 kernel (wgrad_tc.cu) does not apply (the bf16
//     forward and dgrad at these shapes run on tcgen05 + TMEM, conv_tc.cu).
// Replaces SCN's Convolution.cu dConvolution_KMxKN_forward/backward_dW (SURVEY.md 2.2; reference
// call sites src/networks/sparse_building_blocks.py:29-34,110-117,207-213).
#include "common.cuh"

// conv_tc.cu (tcgen05 path)
bool scn_tc_shape_ok(int K, int n_in, int n_out);
size_t scn_tc_image_bytes(int K, int n_in, int n_out, int tf32);
int scn_tc_prep(const float* W, int K, int Cin, int Cout, int transpose, int mirror, int tf32, void* out, cudaStream_t s);
bool scn_stem_tc_shape_ok(int K, int n_in, int n_out);   // stem_tc.cu
int scn_stem_tc_forward(const void* x, int x_dtype, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, const float* W,
                        const float* bias, void* out, int out_dtype, cudaStream_t s);
int scn_stem_tc_wgrad(const void* x, int x_dtype, const void* dout, int dout_dtype, const int32_t* nbr, int K, int64_t n_rows,
                      int64_t n_pad, float* dW, cudaStream_t s);
int scn_wgrad_tc(const void* x, const void* dout, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int Cin, int Cout,
                 int tf32, float* dW, const float* colsum, float* dbias, int accumulate, cudaStream_t s);
int scn_tc_forward(const void* in, int64_t n_in_rows, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int n_in,
                   int n_out, const void* bimg, const float* bias, void* out, int tf32, cudaStream_t s);

namespace {

// =============================================================================================
// weight preparation
// =============================================================================================
// layout 0 (generic kernels): B[k][c][n] fp32, n fastest.  layout 1 (mma): Bt[k][n][c] bf16, c fastest.
template <typename TOut, int LAYOUT>
__global__ void k_prep_weights(const float* __restrict__ W, int K, int Cin, int Cout, int transpose, int mirror,
                               TOut* __restrict__ out) {
  int64_t total = (int64_t)K * Cin * Cout;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int n_in = transpose ? Cout : Cin, n_out = transpose ? Cin : Cout;
  int k = (int)(i / ((int64_t)n_in * n_out));
  int rem = (int)(i - (int64_t)k * n_in * n_out);
  int c, n;
  if (LAYOUT == 0) { c = rem / n_out; n = rem % n_out; } else { n = rem / n_in; c = rem % n_in; }
  int src_k = (transpose && mirror) ? K - 1 - k : k;
  int ci = transpose ? n : c, co = transpose ? c : n;
  float v = W[((int64_t)src_k * Cin + ci) * Cout + co];
  Elem<TOut>::st(out + i, v);
}

// =============================================================================================
// exact fp32 kernels
// =============================================================================================
template <typename TI, typename TO>
__global__ void k_conv_generic(const TI* __restrict__ in, const int32_t* __restrict__ nbr, int K, int64_t n_rows,
                               int64_t n_pad, int n_in, int n_out, const float* __restrict__ B,
                               const float* __restrict__ bias, TO* __restrict__ out) {
  int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= n_rows * n_out) return;
  int64_t o = idx / n_out;
  int n = (int)(idx - o * n_out);
  float acc = bias ? bias[n] : 0.f;
  for (int k = 0; k < K; ++k) {
    int j = nbr[(int64_t)k * n_pad + o];
    if (j < 0) continue;
    const TI* xr = in + (int64_t)j * n_in;
    const float* b = B + (int64_t)k * n_in * n_out + n;
    for (int c = 0; c < n_in; ++c) acc = fmaf(Elem<TI>::ld(xr + c), b[(int64_t)c * n_out], acc);
  }
  Elem<TO>::st(out + idx, acc);
}

// Single input channel (the 5x5x5 / 1x5x5 stem, reference src/networks/resnet.py:30-36,44-50): a K-tap stencil on
// a scalar field -- pure bandwidth.  One thread per output row keeps all NOUT accumulators in registers, reads its
// K neighbour indices (coalesced across the warp) and the weights from shared memory (broadcast).
template <typename TI, typename TO, int NOUT>
__global__ void __launch_bounds__(256) k_conv_cin1(const TI* __restrict__ in, const int32_t* __restrict__ nbr, int K,
                                                   int64_t n_rows, int64_t n_pad, const float* __restrict__ B,
                                                   const float* __restrict__ bias, TO* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float s_w[];          // [K][NOUT]
  for (int i = threadIdx.x; i < K * NOUT; i += blockDim.x) s_w[i] = B[i];
  __syncthreads();
  const int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (o >= n_rows) return;
  float acc[NOUT];
#pragma unroll
  for (int c = 0; c < NOUT; ++c) acc[c] = bias ? bias[c] : 0.f;
  int j = nbr[o];
  for (int k = 0; k < K; ++k) {
    const int jn = k + 1 < K ? nbr[(int64_t)(k + 1) * n_pad + o] : -1;
    if (j >= 0) {
      const float v = Elem<TI>::ld(in + j);
      const float* w = s_w + k * NOUT;
#pragma unroll
      for (int c = 0; c < NOUT; ++c) acc[c] = fmaf(v, w[c], acc[c]);
    }
    j = jn;
  }
  TO* dst = out + o * NOUT;
#pragma unroll
  for (int c = 0; c < NOUT; c += 4) st4(dst + c, make_float4(acc[c], acc[c + 1], acc[c + 2], acc[c + 3]));
}

// dW[k][c][n] += sum over rows o of the chunk with nbr[k][o] >= 0 of in[nbr][c] * dout[o][n]
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) k_wgrad_generic(const TI* __restrict__ in, const TO* __restrict__ dout,
                                                       const int32_t* __restrict__ nbr, int64_t n_rows, int64_t n_pad,
                                                       int n_in, int n_out, int chunk, float* __restrict__ dW) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ int s_list[];   // compacted (in,out) pairs of this chunk: [2][chunk]
  __shared__ int s_count;
  const int k = blockIdx.y;
  const int64_t r0 = (int64_t)blockIdx.x * chunk;
  if (threadIdx.x == 0) s_count = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < chunk; i += blockDim.x) {
    int64_t o = r0 + i;
    if (o < n_rows) {
      int j = nbr[(int64_t)k * n_pad + o];
      if (j >= 0) {
        int p = atomicAdd(&s_count, 1);
        s_list[p] = j;
        s_list[chunk + p] = (int)o;
      }
    }
  }
  __syncthreads();
  const int cnt = s_count;
  if (cnt == 0) return;
  const int total = n_in * n_out;
  for (int e = threadIdx.x; e < total; e += blockDim.x) {
    int c = e / n_out, n = e - c * n_out;
    float acc = 0.f;
    for (int p = 0; p < cnt; ++p)
      acc = fmaf(Elem<TI>::ld(in + (int64_t)s_list[p] * n_in + c), Elem<TO>::ld(dout + (int64_t)s_list[chunk + p] * n_out + n), acc);
    atomicAdd(dW + ((int64_t)k * n_in + c) * n_out + n, acc);
  }
}

// =============================================================================================
// mma.sync helpers
// =============================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(src), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x2_trans(uint32_t addr, uint32_t& r0, uint32_t& r1) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];\n" : "=r"(r0), "=r"(r1) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float* d, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// Copies 8 consecutive channels of a feature row (or zeros when row < 0) to 16 bytes of smem as bf16.
template <typename T> struct RowChunk;
template <> struct RowChunk<__nv_bfloat16> {
  static __device__ __forceinline__ void copy(__nv_bfloat16* dst, const __nv_bfloat16* base, int64_t row, int stride,
                                              int col) {
    const __nv_bfloat16* src = row >= 0 ? base + row * stride + col : base;
    cp_async16(smem_u32(dst), src, row >= 0 ? 16 : 0);
  }
};
template <> struct RowChunk<float> {
  static __device__ __forceinline__ void copy(__nv_bfloat16* dst, const float* base, int64_t row, int stride, int col) {
    uint4 u = make_uint4(0, 0, 0, 0);
    if (row >= 0) {
      const float4* p = reinterpret_cast<const float4*>(base + row * stride + col);
      float4 a = __ldg(p), b = __ldg(p + 1);
      u.x = pack_bf16x2(a.x, a.y); u.y = pack_bf16x2(a.z, a.w);
      u.z = pack_bf16x2(b.x, b.y); u.w = pack_bf16x2(b.z, b.w);
    }
    *reinterpret_cast<uint4*>(dst) = u;
  }
};

// =============================================================================================
// forward / dgrad: out[o, n0:n0+NT] = bias + sum_k in[nbr[k][o], :] . Bt[k][n0:n0+NT, :]^T
// CTA = 4 warps, tile 64 output rows x NT columns, whole n_in (<= 256) contracted per offset,
// 2-stage cp.async pipeline over the offsets that are live in this tile.
// =============================================================================================
constexpr int kBM = 64;

template <typename T, int NT>
__global__ void __launch_bounds__(128) k_conv_mma(const T* __restrict__ in, const int32_t* __restrict__ nbr, int K,
                                                  int64_t n_rows, int64_t n_pad, int n_in, int n_out,
                                                  const __nv_bfloat16* __restrict__ Bt, const float* __restrict__ bias,
                                                  T* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lda = n_in + 8;
  int* s_nbr = reinterpret_cast<int*>(smem_raw);                       // [K][64]
  int* s_klist = s_nbr + K * kBM;                                      // [K]
  int* s_flag = s_klist + K;                                           // [K]
  __shared__ int s_nk;
  size_t off = (size_t)((K * kBM + 2 * K) * sizeof(int) + 15) / 16 * 16;
  __nv_bfloat16* sA = reinterpret_cast<__nv_bfloat16*>(smem_raw + off);          // [2][64][lda]
  __nv_bfloat16* sB = sA + 2 * kBM * lda;                                        // [2][NT][lda]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t row_base = (int64_t)blockIdx.x * kBM;
  const int n0 = blockIdx.y * NT;

  for (int i = tid; i < K * kBM; i += 128) {
    int k = i / kBM, r = i - k * kBM;
    s_nbr[i] = nbr[(int64_t)k * n_pad + row_base + r];
  }
  __syncthreads();
  for (int k = tid; k < K; k += 128) {
    int any = 0;
    for (int r = 0; r < kBM; ++r) any |= (s_nbr[k * kBM + ((r + k) & (kBM - 1))] >= 0);
    s_flag[k] = any;
  }
  __syncthreads();
  if (tid == 0) {
    int c = 0;
    for (int k = 0; k < K; ++k)
      if (s_flag[k]) s_klist[c++] = k;
    s_nk = c;
  }
  __syncthreads();
  const int nk = s_nk;

  float acc[NT / 8][4];
#pragma unroll
  for (int j = 0; j < NT / 8; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;

  const int cpr = n_in / 8;
  auto load_stage = [&](int stage, int k) {
    __nv_bfloat16* a = sA + (size_t)stage * kBM * lda;
    for (int c = tid; c < kBM * cpr; c += 128) {
      int r = c / cpr, q = c - r * cpr;
      RowChunk<T>::copy(a + r * lda + q * 8, in, (int64_t)s_nbr[k * kBM + r], n_in, q * 8);
    }
    __nv_bfloat16* b = sB + (size_t)stage * NT * lda;
    const __nv_bfloat16* src = Bt + ((int64_t)k * n_out + n0) * n_in;
    for (int c = tid; c < NT * cpr; c += 128) {
      int r = c / cpr, q = c - r * cpr;
      cp_async16(smem_u32(b + r * lda + q * 8), src + (int64_t)r * n_in + q * 8, 16);
    }
    cp_async_commit();
  };

  if (nk > 0) load_stage(0, s_klist[0]);
  for (int it = 0; it < nk; ++it) {
    const int stage = it & 1;
    if (it + 1 < nk) {
      load_stage(stage ^ 1, s_klist[it + 1]);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const __nv_bfloat16* a = sA + (size_t)stage * kBM * lda + (warp * 16) * lda;
    const __nv_bfloat16* b = sB + (size_t)stage * NT * lda;
    for (int kk = 0; kk < n_in; kk += 16) {
      uint32_t a0, a1, a2, a3;
      ldmatrix_x4(smem_u32(a + (lane & 15) * lda + kk + (lane >> 4) * 8), a0, a1, a2, a3);
#pragma unroll
      for (int jn = 0; jn < NT / 16; ++jn) {
        uint32_t b0, b1, b2, b3;
        const int nrow = jn * 16 + (lane >> 4) * 8 + (lane & 7);
        ldmatrix_x4(smem_u32(b + nrow * lda + kk + ((lane >> 3) & 1) * 8), b0, b1, b2, b3);
        mma_bf16(acc[2 * jn], a0, a1, a2, a3, b0, b1);
        mma_bf16(acc[2 * jn + 1], a0, a1, a2, a3, b2, b3);
      }
    }
    __syncthreads();
  }

  const int g = lane >> 2, t = lane & 3;
  const int64_t r_lo = row_base + warp * 16 + g, r_hi = r_lo + 8;
#pragma unroll
  for (int j = 0; j < NT / 8; ++j) {
    const int col = n0 + j * 8 + 2 * t;
    const float b0 = bias ? bias[col] : 0.f, b1 = bias ? bias[col + 1] : 0.f;
    if (r_lo < n_rows) {
      Elem<T>::st(out + r_lo * n_out + col, acc[j][0] + b0);
      Elem<T>::st(out + r_lo * n_out + col + 1, acc[j][1] + b1);
    }
    if (r_hi < n_rows) {
      Elem<T>::st(out + r_hi * n_out + col, acc[j][2] + b0);
      Elem<T>::st(out + r_hi * n_out + col + 1, acc[j][3] + b1);
    }
  }
}

// =============================================================================================
// wgrad: dW[k][:, n0:n0+NT] += sum over live pairs of the chunk  in[pi, :]^T . dout[po, n0:n0+NT]
// CTA = 8 warps (2 along n_in x 4 along NT); pairs are compacted from nbr[k][chunk] on the fly,
// consumed 64 at a time; both operands reach the MMA through ldmatrix.trans.
// =============================================================================================
constexpr int kPB = 64;        // pairs per MMA step
constexpr int kScan = 256;     // rows scanned per compaction pass (= threads)
constexpr int kMaxChunk = 4096;   // rows per CTA: bounds the shared-memory pair list (worst case: every row is a pair)

template <typename T, int MI, int NJ>
__global__ void __launch_bounds__(256) k_wgrad_mma(const T* __restrict__ in, const T* __restrict__ dout,
                                                   const int32_t* __restrict__ nbr, int64_t n_rows, int64_t n_pad,
                                                   int n_out, int chunk, float* __restrict__ dW) {
  constexpr int n_in = 32 * MI, NT = 32 * NJ;
  constexpr int lda = n_in + 8, ldb = NT + 8;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __nv_bfloat16* sA = reinterpret_cast<__nv_bfloat16*>(smem_raw);   // [2][kPB][lda]
  __nv_bfloat16* sB = sA + 2 * kPB * lda;                           // [2][kPB][ldb]
  int* s_in = reinterpret_cast<int*>(sB + 2 * kPB * ldb);           // [chunk]
  int* s_out = s_in + chunk;                                        // [chunk]
  __shared__ int s_warp_cnt[8];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp & 1, wn = warp >> 1;
  const int k = blockIdx.y;
  const int n0 = blockIdx.z * NT;
  const int64_t r0 = (int64_t)blockIdx.x * chunk;
  const int64_t r1 = r0 + chunk < n_rows ? r0 + chunk : n_rows;

  // ---- phase A: compact the live (in,out) pairs of offset k in this chunk (order = out row) -----------------
  int count = 0;
  for (int64_t rb = r0; rb < r1; rb += kScan) {
    const int64_t o = rb + tid;
    int j = -1;
    if (o < r1) j = nbr[(int64_t)k * n_pad + o];
    const unsigned m = __ballot_sync(0xffffffffu, j >= 0);
    if (lane == 0) s_warp_cnt[warp] = __popc(m);
    __syncthreads();
    int base = count, total = count;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      const int c = s_warp_cnt[w];
      if (w < warp) base += c;
      total += c;
    }
    if (j >= 0) {
      const int p = base + __popc(m & ((1u << lane) - 1u));
      s_in[p] = j;
      s_out[p] = (int)o;
    }
    count = total;
    __syncthreads();
  }
  if (count == 0) return;

  float acc[MI][NJ][4];
#pragma unroll
  for (int i = 0; i < MI; ++i)
#pragma unroll
    for (int j = 0; j < NJ; ++j) acc[i][j][0] = acc[i][j][1] = acc[i][j][2] = acc[i][j][3] = 0.f;

  // ---- phase B: double-buffered gather (cp.async) + mma.sync over 64 pairs at a time -------------------------
  const int nsteps = (count + kPB - 1) / kPB;
  auto gather = [&](int step, int buf) {
    const int head = step * kPB;
    const int take = count - head < kPB ? count - head : kPB;
    __nv_bfloat16* a = sA + (size_t)buf * kPB * lda;
    __nv_bfloat16* b = sB + (size_t)buf * kPB * ldb;
    for (int c = tid; c < kPB * (n_in / 8); c += 256) {
      const int r = c / (n_in / 8), q = c - r * (n_in / 8);
      const int64_t row = r < take ? (int64_t)s_in[head + r] : -1;
      RowChunk<T>::copy(a + r * lda + q * 8, in, row, n_in, q * 8);
    }
    for (int c = tid; c < kPB * (NT / 8); c += 256) {
      const int r = c / (NT / 8), q = c - r * (NT / 8);
      const int64_t row = r < take ? (int64_t)s_out[head + r] : -1;
      RowChunk<T>::copy(b + r * ldb + q * 8, dout + n0, row, n_out, q * 8);
    }
    cp_async_commit();
  };
  gather(0, 0);
  for (int s = 0; s < nsteps; ++s) {
    if (s + 1 < nsteps) {
      gather(s + 1, (s + 1) & 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const __nv_bfloat16* a = sA + (size_t)(s & 1) * kPB * lda;
    const __nv_bfloat16* b = sB + (size_t)(s & 1) * kPB * ldb;
#pragma unroll
    for (int kk = 0; kk < kPB; kk += 16) {
      uint32_t bf[NJ][2];
#pragma unroll
      for (int j = 0; j < NJ; ++j)
        ldmatrix_x2_trans(smem_u32(b + (kk + (lane & 15)) * ldb + (wn * NJ + j) * 8), bf[j][0], bf[j][1]);
#pragma unroll
      for (int i = 0; i < MI; ++i) {
        uint32_t a0, a1, a2, a3;
        const int m0 = (wm * MI + i) * 16;
        ldmatrix_x4_trans(smem_u32(a + (kk + (lane >> 4) * 8 + (lane & 7)) * lda + m0 + ((lane >> 3) & 1) * 8), a0, a1,
                          a2, a3);
#pragma unroll
        for (int j = 0; j < NJ; ++j) mma_bf16(acc[i][j], a0, a1, a2, a3, bf[j][0], bf[j][1]);
      }
    }
    __syncthreads();
  }

  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int i = 0; i < MI; ++i)
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int m = (wm * MI + i) * 16 + g;
      const int n = n0 + (wn * NJ + j) * 8 + 2 * t;
      float* d = dW + ((int64_t)k * n_in + m) * n_out + n;
      if (acc[i][j][0] != 0.f) atomicAdd(d, acc[i][j][0]);
      if (acc[i][j][1] != 0.f) atomicAdd(d + 1, acc[i][j][1]);
      if (acc[i][j][2] != 0.f) atomicAdd(d + (int64_t)8 * n_out, acc[i][j][2]);
      if (acc[i][j][3] != 0.f) atomicAdd(d + (int64_t)8 * n_out + 1, acc[i][j][3]);
    }
}

// ---------------------------------------------------------------------------------------------
bool mma_ok(int K, int n_in, int n_out, int precision) {
  return precision == SCN_PREC_BF16 && (n_in % 32) == 0 && (n_out % 32) == 0 && n_in <= 256 && n_out <= 256 &&
         K <= 128;
}
int pick_nt(int n_out) { return (n_out % 64) == 0 ? 64 : ((n_out % 96) == 0 ? 96 : 32); }

template <typename T, int NT>
int launch_conv_mma(const T* in, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int n_in, int n_out,
                    const __nv_bfloat16* Bt, const float* bias, T* out, cudaStream_t s) {
  size_t smem = (size_t)((K * kBM + 2 * K) * sizeof(int) + 15) / 16 * 16 +
                (size_t)(2 * kBM + 2 * NT) * (n_in + 8) * sizeof(__nv_bfloat16);
  auto kern = k_conv_mma<T, NT>;
  SCN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((unsigned)((n_rows + kBM - 1) / kBM), (unsigned)(n_out / NT));
  kern<<<grid, 128, smem, s>>>(in, nbr, K, n_rows, n_pad, n_in, n_out, Bt, bias, out);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

template <typename T>
int conv_mma_t(const T* in, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int n_in, int n_out,
               const __nv_bfloat16* Bt, const float* bias, T* out, cudaStream_t s) {
  switch (pick_nt(n_out)) {
    case 64: return launch_conv_mma<T, 64>(in, nbr, K, n_rows, n_pad, n_in, n_out, Bt, bias, out, s);
    case 96: return launch_conv_mma<T, 96>(in, nbr, K, n_rows, n_pad, n_in, n_out, Bt, bias, out, s);
    default: return launch_conv_mma<T, 32>(in, nbr, K, n_rows, n_pad, n_in, n_out, Bt, bias, out, s);
  }
}

template <typename T, int MI, int NJ>
int launch_wgrad_mma(const T* in, const T* dout, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int n_out,
                     float* dW, cudaStream_t s) {
  constexpr int n_in = 32 * MI, NT = 32 * NJ;
  const int nz = n_out / NT;
  int64_t want = (int64_t)kNumSMs * 8 / ((int64_t)K * nz);
  if (want < 1) want = 1;
  int64_t chunk = round_up_i64((n_rows + want - 1) / want, kScan);
  if (chunk > kMaxChunk) chunk = kMaxChunk;
  size_t smem = (size_t)2 * kPB * (n_in + 8 + NT + 8) * sizeof(__nv_bfloat16) + 2 * (size_t)chunk * sizeof(int);
  auto kern = k_wgrad_mma<T, MI, NJ>;
  SCN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((unsigned)((n_rows + chunk - 1) / chunk), (unsigned)K, (unsigned)nz);
  kern<<<grid, 256, smem, s>>>(in, dout, nbr, n_rows, n_pad, n_out, (int)chunk, dW);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

template <typename T, int MI>
int wgrad_mma_mi(const T* in, const T* dout, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int n_out,
                 float* dW, cudaStream_t s) {
  switch (pick_nt(n_out)) {
    case 64: return launch_wgrad_mma<T, MI, 2>(in, dout, nbr, K, n_rows, n_pad, n_out, dW, s);
    case 96: return launch_wgrad_mma<T, MI, 3>(in, dout, nbr, K, n_rows, n_pad, n_out, dW, s);
    default: return launch_wgrad_mma<T, MI, 1>(in, dout, nbr, K, n_rows, n_pad, n_out, dW, s);
  }
}

template <typename T>
int wgrad_mma_t(const T* in, const T* dout, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int n_in,
                int n_out, float* dW, cudaStream_t s) {
  switch (n_in / 32) {
    case 1: return wgrad_mma_mi<T, 1>(in, dout, nbr, K, n_rows, n_pad, n_out, dW, s);
    case 2: return wgrad_mma_mi<T, 2>(in, dout, nbr, K, n_rows, n_pad, n_out, dW, s);
    case 3: return wgrad_mma_mi<T, 3>(in, dout, nbr, K, n_rows, n_pad, n_out, dW, s);
    case 4: return wgrad_mma_mi<T, 4>(in, dout, nbr, K, n_rows, n_pad, n_out, dW, s);
    case 5: return wgrad_mma_mi<T, 5>(in, dout, nbr, K, n_rows, n_pad, n_out, dW, s);
    case 6: return wgrad_mma_mi<T, 6>(in, dout, nbr, K, n_rows, n_pad, n_out, dW, s);
    case 7: return wgrad_mma_mi<T, 7>(in, dout, nbr, K, n_rows, n_pad, n_out, dW, s);
    case 8: return wgrad_mma_mi<T, 8>(in, dout, nbr, K, n_rows, n_pad, n_out, dW, s);
    default: return SCN_ERR_UNSUPPORTED;
  }
}

template <typename TI, typename TO>
int conv_generic_t(const TI* in, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int n_in, int n_out,
                   const float* B, const float* bias, TO* out, cudaStream_t s) {
  if (n_in == 1 && (n_out == 16 || n_out == 32 || n_out == 64) && (size_t)K * n_out * 4 <= 48 * 1024) {
    const size_t smem = (size_t)K * n_out * sizeof(float);
    const unsigned g = grid_for(n_rows, 256);
    if (n_out == 16) SCN_CUDA(scn_launch_pdl(k_conv_cin1<TI, TO, 16>, dim3(g), dim3(256), smem, s, in, nbr, K, n_rows, n_pad, B, bias, out));
    else if (n_out == 32) SCN_CUDA(scn_launch_pdl(k_conv_cin1<TI, TO, 32>, dim3(g), dim3(256), smem, s, in, nbr, K, n_rows, n_pad, B, bias, out));
    else SCN_CUDA(scn_launch_pdl(k_conv_cin1<TI, TO, 64>, dim3(g), dim3(256), smem, s, in, nbr, K, n_rows, n_pad, B, bias, out));
    SCN_LAUNCH_CHECK();
    return SCN_OK;
  }
  k_conv_generic<TI, TO><<<grid_for(n_rows * n_out, 256), 256, 0, s>>>(in, nbr, K, n_rows, n_pad, n_in, n_out, B, bias,
                                                                       out);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

template <typename TI, typename TO>
int wgrad_generic_t(const TI* in, const TO* dout, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int n_in,
                    int n_out, float* dW, cudaStream_t s) {
  const int chunk = 512;
  dim3 grid((unsigned)((n_rows + chunk - 1) / chunk), (unsigned)K);
  SCN_CUDA(scn_launch_pdl(k_wgrad_generic<TI, TO>, grid, dim3(256), 2 * chunk * sizeof(int), s, in, dout, nbr, n_rows, n_pad, n_in,
                          n_out, chunk, dW));
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

}  // namespace

// 0: exact fp32 FMA kernels; 1: mma.sync (HMMA) kernels, Bt[k][n][c] bf16; 2: tcgen05 kernel, swizzled image (bf16
// features with SCN_PREC_BF16, fp32 features with SCN_PREC_TF32)
static int conv_path(int K, int n_in, int n_out, int precision, int feat_dtype) {
  const bool tc_mode = (precision == SCN_PREC_BF16 && feat_dtype == SCN_BF16) ||
                       (precision == SCN_PREC_TF32 && feat_dtype == SCN_F32);
  if (tc_mode && scn_tc_shape_ok(K, n_in, n_out)) return 2;
  return mma_ok(K, n_in, n_out, precision) ? 1 : 0;
}
// the tcgen05 path of a precision runs its TF32 instantiation
static int tc_tf32(int precision) { return precision == SCN_PREC_TF32 ? 1 : 0; }

extern "C" int scn_conv_path(int K, int n_in, int n_out, int precision, int feat_dtype) {
  return conv_path(K, n_in, n_out, precision, feat_dtype);
}

extern "C" size_t scn_conv_prep_bytes(int K, int n_in, int n_out, int precision, int feat_dtype) {
  switch (conv_path(K, n_in, n_out, precision, feat_dtype)) {
    case 2: return scn_tc_image_bytes(K, n_in, n_out, tc_tf32(precision));
    case 1: return (size_t)K * n_in * n_out * 2;
    default: return (size_t)K * n_in * n_out * 4;
  }
}

extern "C" int scn_conv_prep_weights(const float* W, int K, int Cin, int Cout, int transpose, int mirror,
                                     int precision, int feat_dtype, void* out, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (!W || !out || K < 1 || Cin < 1 || Cout < 1) return SCN_ERR_ARG;
  const int n_in = transpose ? Cout : Cin, n_out = transpose ? Cin : Cout;
  int64_t total = (int64_t)K * Cin * Cout;
  unsigned g = grid_for(total, 256);
  const int path = conv_path(K, n_in, n_out, precision, feat_dtype);
  if (path == 2) return scn_tc_prep(W, K, Cin, Cout, transpose, mirror, tc_tf32(precision), out, s);
  if (path == 1)
    k_prep_weights<__nv_bfloat16, 1><<<g, 256, 0, s>>>(W, K, Cin, Cout, transpose, mirror, (__nv_bfloat16*)out);
  else
    k_prep_weights<float, 0><<<g, 256, 0, s>>>(W, K, Cin, Cout, transpose, mirror, (float*)out);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

extern "C" int scn_conv_forward(const void* in, int in_dtype, int64_t n_in_rows, const int32_t* nbr, int K,
                                int64_t n_out_rows, int64_t n_pad, int n_in, int n_out, const void* Bprep,
                                const float* bias, int precision, void* out, int out_dtype, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n_out_rows == 0) return SCN_OK;
  if (!in || !nbr || !Bprep || !out || K < 1 || n_pad < n_out_rows || (n_pad & 127)) return SCN_ERR_ARG;
  if (precision == SCN_PREC_FP32 && (in_dtype != SCN_F32 || out_dtype != SCN_F32)) return SCN_ERR_ARG;
  if (in_dtype == out_dtype && conv_path(K, n_in, n_out, precision, in_dtype) == 2)
    return scn_tc_forward(in, n_in_rows, nbr, K, n_out_rows, n_pad, n_in, n_out, Bprep, bias, out, tc_tf32(precision), s);
  if (mma_ok(K, n_in, n_out, precision) && in_dtype == out_dtype) {
    // fp32 features of the "mixed" mode (bf16 features at these shapes took the tcgen05 path above)
    if (in_dtype == SCN_F32)
      return conv_mma_t<float>((const float*)in, nbr, K, n_out_rows, n_pad, n_in, n_out, (const __nv_bfloat16*)Bprep,
                               bias, (float*)out, s);
    return SCN_ERR_ARG;
  }
  if (mma_ok(K, n_in, n_out, precision)) return SCN_ERR_UNSUPPORTED;   // Bprep is bf16 for this shape
  const float* B = (const float*)Bprep;
  // the stem (one input channel) as a dense GEMM over the neighbour table on tensor cores (stem_tc.cu): bf16 outputs,
  // and fp32 outputs in the tf32 mode; the exact fp32 mode keeps the FFMA kernel
  if (precision != SCN_PREC_FP32 && (out_dtype == SCN_BF16 || precision == SCN_PREC_TF32) &&
      scn_stem_tc_shape_ok(K, n_in, n_out))
    return scn_stem_tc_forward(in, in_dtype, nbr, K, n_out_rows, n_pad, B, bias, out, out_dtype, s);
  if (in_dtype == SCN_F32 && out_dtype == SCN_F32)
    return conv_generic_t<float, float>((const float*)in, nbr, K, n_out_rows, n_pad, n_in, n_out, B, bias, (float*)out, s);
  if (in_dtype == SCN_F32 && out_dtype == SCN_BF16)
    return conv_generic_t<float, __nv_bfloat16>((const float*)in, nbr, K, n_out_rows, n_pad, n_in, n_out, B, bias,
                                                (__nv_bfloat16*)out, s);
  if (in_dtype == SCN_BF16 && out_dtype == SCN_F32)
    return conv_generic_t<__nv_bfloat16, float>((const __nv_bfloat16*)in, nbr, K, n_out_rows, n_pad, n_in, n_out, B,
                                                bias, (float*)out, s);
  if (in_dtype == SCN_BF16 && out_dtype == SCN_BF16)
    return conv_generic_t<__nv_bfloat16, __nv_bfloat16>((const __nv_bfloat16*)in, nbr, K, n_out_rows, n_pad, n_in,
                                                        n_out, B, bias, (__nv_bfloat16*)out, s);
  return SCN_ERR_ARG;
}

// scn_conv_wgrad that also adds dbias[n_out] (+)= colsum (accumulate_dbias) when colsum != NULL and the tcgen05 path can
// fold it into its reduction kernel; *bias_folded tells whether it did (otherwise the caller adds it: module_api.cu).
int scn_conv_wgrad_fold(const void* in, int in_dtype, const void* dout, int dout_dtype, const int32_t* nbr, int K,
                        int64_t n_rows, int64_t n_pad, int n_in, int n_out, int precision, float* dW, const float* colsum,
                        float* dbias, int accumulate_dbias, bool* bias_folded, cudaStream_t s) {
  *bias_folded = false;
  if (n_rows == 0) return SCN_OK;
  if (!in || !dout || !nbr || !dW || K < 1 || n_pad < n_rows) return SCN_ERR_ARG;
  if (precision == SCN_PREC_FP32 && (in_dtype != SCN_F32 || dout_dtype != SCN_F32)) return SCN_ERR_ARG;
  const bool tc_bf16 = precision == SCN_PREC_BF16 && in_dtype == SCN_BF16 && dout_dtype == SCN_BF16;
  const bool tc_tf = precision == SCN_PREC_TF32 && in_dtype == SCN_F32 && dout_dtype == SCN_F32;
  if ((tc_bf16 || tc_tf) && (n_pad & 127) == 0) {
    // tcgen05 path.  The number of rows of `in` is not part of this entry point's signature; the kernel addresses
    // gathered rows through 32-bit offsets in 16-byte units, i.e. feature matrices up to 64 GB.
    int rc = scn_wgrad_tc(in, dout, nbr, K, n_rows, n_pad, n_in, n_out, tc_tf ? 1 : 0, dW, colsum, dbias,
                          accumulate_dbias, s);
    *bias_folded = rc == SCN_OK && colsum != nullptr;
    if (rc != SCN_ERR_UNSUPPORTED) return rc;
  }
  // the stem (one input channel): dense GEMM over the neighbour table on tensor cores (stem_tc.cu); bf16 dout, and fp32
  // dout in the tf32 mode
  if (precision != SCN_PREC_FP32 && (dout_dtype == SCN_BF16 || precision == SCN_PREC_TF32) && (n_pad & 127) == 0 &&
      scn_stem_tc_shape_ok(K, n_in, n_out))
    return scn_stem_tc_wgrad(in, in_dtype, dout, dout_dtype, nbr, K, n_rows, n_pad, dW, s);
  if (mma_ok(K, n_in, n_out, precision) && in_dtype == dout_dtype) {
    if (in_dtype == SCN_F32)
      return wgrad_mma_t<float>((const float*)in, (const float*)dout, nbr, K, n_rows, n_pad, n_in, n_out, dW, s);
    if (in_dtype == SCN_BF16)
      return wgrad_mma_t<__nv_bfloat16>((const __nv_bfloat16*)in, (const __nv_bfloat16*)dout, nbr, K, n_rows, n_pad,
                                        n_in, n_out, dW, s);
    return SCN_ERR_ARG;
  }
  if (in_dtype == SCN_F32 && dout_dtype == SCN_F32)
    return wgrad_generic_t<float, float>((const float*)in, (const float*)dout, nbr, K, n_rows, n_pad, n_in, n_out, dW, s);
  if (in_dtype == SCN_F32 && dout_dtype == SCN_BF16)
    return wgrad_generic_t<float, __nv_bfloat16>((const float*)in, (const __nv_bfloat16*)dout, nbr, K, n_rows, n_pad,
                                                 n_in, n_out, dW, s);
  if (in_dtype == SCN_BF16 && dout_dtype == SCN_F32)
    return wgrad_generic_t<__nv_bfloat16, float>((const __nv_bfloat16*)in, (const float*)dout, nbr, K, n_rows, n_pad,
                                                 n_in, n_out, dW, s);
  if (in_dtype == SCN_BF16 && dout_dtype == SCN_BF16)
    return wgrad_generic_t<__nv_bfloat16, __nv_bfloat16>((const __nv_bfloat16*)in, (const __nv_bfloat16*)dout, nbr, K,
                                                         n_rows, n_pad, n_in, n_out, dW, s);
  return SCN_ERR_ARG;
}

extern "C" int scn_conv_wgrad(const void* in, int in_dtype, const void* dout, int dout_dtype, const int32_t* nbr,
                              int K, int64_t n_rows, int64_t n_pad, int n_in, int n_out, int precision, float* dW,
                              void* stream) {
  bool bias_folded;
  return scn_conv_wgrad_fold(in, in_dtype, dout, dout_dtype, nbr, K, n_rows, n_pad, n_in, n_out, precision, dW, nullptr,
                             nullptr, 0, &bias_folded, (cudaStream_t)stream);
}
