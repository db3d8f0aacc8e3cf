// Stem convolution (one input channel, 5^3 or 1x5x5 filter, 32 output channels) on tensor cores.
//     forward:  out[o, :] = bias + sum_k x[nbr[k][o]] * W[k][:]
//     wgrad:    dW[k][:] += sum_o x[nbr[k][o]] * dout[o, :]
// With a scalar input feature the gather-GEMM of the other layers degenerates: the first-generation kernels
// (conv.cu::k_conv_cin1, k_wgrad_generic) spend one FFMA per (row, offset, output channel) although only ~16% of the
// 125 neighbours of a site exist -- 262 us forward + 381 us wgrad per step at 495 k rows, ~6x the table's HBM time.
// Here both are DENSE GEMMs over the neighbour TABLE on mma.sync (m16n8k16, bf16 x bf16 -> fp32): the matrix
// A[o][k] = x[nbr[k][o]] (0 where there is no neighbour) is built in registers straight from the table, in exactly the
// fragment layout the instruction wants, so a missing neighbour costs nothing but its table entry:
//     forward:  out[16 rows x 32]  = A[16 x 128] . W[128 x 32]        (K = 125 padded to 128)
//     wgrad:    dW[128 x 32]      += A^T[128 x 16 rows] . dout[16 rows x 32]
// Precision: x and W are fp32 in HBM; each is split into bf16 hi + lo parts (x = hi + lo to 2^-17) and the products
// hi.hi + lo.hi + hi.lo are accumulated in fp32, i.e. ~fp32 accuracy (the lo.lo term is below 2^-16 relative); dout is
// bf16 already in the "bf16" mode.  In the "tf32" mode (fp32 features) the output is stored fp32 and the fp32 dout of
// the weight gradient is split like x: hi.hi + lo.hi + hi.lo.  Used in the "bf16", "mixed" (bf16 outputs only) and
// "tf32" precision modes; the "fp32" mode keeps the exact FFMA kernels.
// HBM-bound by the table (4 K n bytes: 248 MB for the bench batch).
//
// Replaces SCN's Convolution forward / backward for the reference's initial_convolution
// (src/networks/resnet.py:30-36: SubmanifoldConvolution(nIn=1, nOut=n_initial_filters, filter_size=5)).
#include <type_traits>

#include "common.cuh"

namespace stem {

constexpr int NOUT = 32;
constexpr int MAXKT = 8;                 // K <= 128

__device__ __forceinline__ void mma16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// (v0, v1) -> bf16x2 of the rounded values (hi) and of the remainders (lo); the first value in the low half
__device__ __forceinline__ void split2(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
  __nv_bfloat162 h;
  h.x = h0; h.y = h1;
  hi = *reinterpret_cast<uint32_t*>(&h);
  lo = pack_bf16x2(v0 - __bfloat162float(h0), v1 - __bfloat162float(h1));
}
__device__ __forceinline__ float ldx(const float* x, int j) { return j >= 0 ? __ldg(x + j) : 0.f; }
__device__ __forceinline__ float ldx(const __nv_bfloat16* x, int j) { return j >= 0 ? __bfloat162float(x[j]) : 0.f; }
// two adjacent output values of a row: bf16x2 or float2
__device__ __forceinline__ void st2(__nv_bfloat16* p, float a, float b) { *reinterpret_cast<uint32_t*>(p) = pack_bf16x2(a, b); }
__device__ __forceinline__ void st2(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
// one element of dout as the raw bf16 bits (bf16 dout) or as fp32
__device__ __forceinline__ unsigned short ldd(const __nv_bfloat16* d, int64_t i) {
  return reinterpret_cast<const unsigned short*>(d)[i];
}
__device__ __forceinline__ float ldd(const float* d, int64_t i) { return d[i]; }

// Forward.  One warp per 16-row tile (grid-stride); thread (g = lane / 4, t = lane % 4) of the m16n8k16 layout holds
// A[g | g + 8][2t, 2t + 1, 2t + 8, 2t + 9] of every 16-offset block: eight table entries, eight gathered scalars.
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) k_stem_fwd(const TI* __restrict__ x, const int32_t* __restrict__ nbr, int K, int64_t n_rows,
                                                  int64_t n_pad, const float* __restrict__ W, const float* __restrict__ bias,
                                                  TO* __restrict__ out) {
  __shared__ uint2 s_bhi[MAXKT * 4 * 32], s_blo[MAXKT * 4 * 32];     // B fragments of (offset block, 8-column block, lane)
  pdl_launch_dependents();
  pdl_wait();
  const int nkt = (K + 15) >> 4;
  for (int i = threadIdx.x; i < nkt * 4 * 32; i += blockDim.x) {
    const int lane = i & 31, nt = (i >> 5) & 3, kt = i >> 7;
    const int g = lane >> 2, t = lane & 3, n = nt * 8 + g, k0 = kt * 16 + 2 * t;
    float w[4];
    const int ks[4] = {k0, k0 + 1, k0 + 8, k0 + 9};
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = ks[j] < K ? W[ks[j] * NOUT + n] : 0.f;
    uint2 hi, lo;
    split2(w[0], w[1], hi.x, lo.x);
    split2(w[2], w[3], hi.y, lo.y);
    s_bhi[i] = hi;
    s_blo[i] = lo;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int64_t tiles = (n_rows + 15) >> 4;
  for (int64_t tile = (int64_t)blockIdx.x * wpb + warp; tile < tiles; tile += (int64_t)gridDim.x * wpb) {
    const int64_t r0 = tile * 16;
    float acc[4][4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const float b0 = bias ? bias[nt * 8 + 2 * t] : 0.f, b1 = bias ? bias[nt * 8 + 2 * t + 1] : 0.f;
      acc[nt][0] = b0; acc[nt][1] = b1; acc[nt][2] = b0; acc[nt][3] = b1;
    }
    // table entries of the next offset block are in flight while this one is gathered and multiplied
    auto load_idx = [&](int kt, int* idx) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int k = kt * 16 + 2 * t + (j & 1) + (j >> 1) * 8;
        const int32_t* col = nbr + (int64_t)k * n_pad + r0 + g;
        idx[j] = k < K ? __ldg(col) : -1;            // row g
        idx[4 + j] = k < K ? __ldg(col + 8) : -1;    // row g + 8 (n_pad is a multiple of 128: always inside the table)
      }
    };
    int idx[8], nxt[8];
    load_idx(0, idx);
    for (int kt = 0; kt < nkt; ++kt) {
      if (kt + 1 < nkt) load_idx(kt + 1, nxt);
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = ldx(x, idx[j]);
      uint32_t ahi[4], alo[4];
      split2(v[0], v[1], ahi[0], alo[0]);            // row g,     offsets 2t, 2t + 1
      split2(v[4], v[5], ahi[1], alo[1]);            // row g + 8, offsets 2t, 2t + 1
      split2(v[2], v[3], ahi[2], alo[2]);            // row g,     offsets 2t + 8, 2t + 9
      split2(v[6], v[7], ahi[3], alo[3]);            // row g + 8, offsets 2t + 8, 2t + 9
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const uint2 bh = s_bhi[(kt * 4 + nt) * 32 + lane], bl = s_blo[(kt * 4 + nt) * 32 + lane];
        mma16816(acc[nt], ahi, bh.x, bh.y);
        mma16816(acc[nt], alo, bh.x, bh.y);
        mma16816(acc[nt], ahi, bl.x, bl.y);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) idx[j] = nxt[j];
    }
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const int col = nt * 8 + 2 * t;
      if (r0 + g < n_rows) st2(out + (r0 + g) * NOUT + col, acc[nt][0], acc[nt][1]);
      if (r0 + g + 8 < n_rows) st2(out + (r0 + g + 8) * NOUT + col, acc[nt][2], acc[nt][3]);
    }
  }
}

// Weight gradient.  dW^T is never formed: the accumulator is dW[offset][channel] itself, M = offsets (128 = 8 blocks of 16),
// N = 32 channels, contraction over the rows.  A block works on two 16-row tiles at a time (warp / 4) and splits the 128
// offsets over four warps (warp % 4: 32 offsets = 2 blocks each), so a thread holds 2 x 4 accumulator fragments.  The A
// operand is A^T[offset][row]: thread (g, t) needs x[nbr[k][r0 + 2t, 2t + 1 (+ 8)]] for k = g, g + 8 of each offset
// block -- pairs of adjacent table entries, one 8-byte load each.  The B operand dout[row][channel] is read with the
// fragment's own (strided, L1-resident) 2-byte accesses.  Blocks add their partial dW with fp32 atomics at the end
// (one pass of 4 K values per block).  An fp32 dout (tf32 mode) is split into hi + lo fragments like x, and the products
// hi.hi + lo.hi + hi.lo are accumulated.
template <typename TI, typename TD>
__global__ void __launch_bounds__(256, 2) k_stem_wgrad(const TI* __restrict__ x, const TD* __restrict__ dout,
                                                       const int32_t* __restrict__ nbr, int K, int64_t n_rows, int64_t n_pad,
                                                       float* __restrict__ dW) {
  __shared__ float s_part[4][2 * 4 * 4 * 32];              // the second row-tile stream's accumulators, per offset group
  pdl_launch_dependents();
  pdl_wait();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int kg = warp & 3, sg = warp >> 2;
  const int64_t tiles = (n_rows + 15) >> 4;
  float acc[2][4][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
  constexpr bool SPLIT_D = std::is_same<TD, float>::value;
  auto load_idx = [&](int64_t r0, int2* idx) {
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k = kg * 32 + mt * 16 + g + 8 * h;
        const int2* col = reinterpret_cast<const int2*>(nbr + (int64_t)k * n_pad + r0 + 2 * t);
        const int2 none = make_int2(-1, -1);
        idx[mt * 4 + h] = k < K ? __ldg(col) : none;             // rows 2t, 2t + 1
        idx[mt * 4 + 2 + h] = k < K ? __ldg(col + 4) : none;     // rows 2t + 8, 2t + 9
      }
  };
  int64_t tile = (int64_t)blockIdx.x * 2 + sg;
  const int64_t tstride = (int64_t)gridDim.x * 2;
  int2 idx[8], nxt[8];
  if (tile < tiles) load_idx(tile * 16, idx);
  for (; tile < tiles; tile += tstride) {
    const int64_t r0 = tile * 16;
    if (tile + tstride < tiles) load_idx((tile + tstride) * 16, nxt);
    // B fragments: b0 = dout[r0 + 2t, 2t + 1][n], b1 = dout[r0 + 2t + 8, 2t + 9][n], n = 8 nt + g; rows past the end are
    // zeros.  bl: the lo parts of an fp32 dout.
    uint32_t b[4][2], bl[4][2];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int64_t ra = r0 + 2 * t + 8 * h;
        if constexpr (SPLIT_D) {
          const float v0 = ra < n_rows ? ldd(dout, ra * NOUT + nt * 8 + g) : 0.f;
          const float v1 = ra + 1 < n_rows ? ldd(dout, (ra + 1) * NOUT + nt * 8 + g) : 0.f;
          split2(v0, v1, b[nt][h], bl[nt][h]);
        } else {
          const unsigned short lo = ra < n_rows ? ldd(dout, ra * NOUT + nt * 8 + g) : (unsigned short)0;
          const unsigned short hi = ra + 1 < n_rows ? ldd(dout, (ra + 1) * NOUT + nt * 8 + g) : (unsigned short)0;
          b[nt][h] = (uint32_t)lo | ((uint32_t)hi << 16);
          bl[nt][h] = 0u;
        }
      }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      uint32_t ahi[4], alo[4];
      // a0: offset g, rows 2t, 2t+1; a1: offset g + 8, same rows; a2: offset g, rows + 8; a3: offset g + 8, rows + 8
#pragma unroll
      for (int f = 0; f < 4; ++f) {
        const int2 j = idx[mt * 4 + f];
        split2(ldx(x, j.x), ldx(x, j.y), ahi[f], alo[f]);
      }
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        mma16816(acc[mt][nt], ahi, b[nt][0], b[nt][1]);
        mma16816(acc[mt][nt], alo, b[nt][0], b[nt][1]);
        if constexpr (SPLIT_D) mma16816(acc[mt][nt], ahi, bl[nt][0], bl[nt][1]);
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) idx[j] = nxt[j];
  }
  // the two row-tile streams of a block are added in shared memory, then one atomic per (offset, channel) and block
  if (sg == 1) {
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) s_part[kg][((mt * 4 + nt) * 4 + e) * 32 + lane] = acc[mt][nt][e];
  }
  __syncthreads();
  if (sg == 0) {
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float v = acc[mt][nt][e] + s_part[kg][((mt * 4 + nt) * 4 + e) * 32 + lane];
          const int k = kg * 32 + mt * 16 + g + ((e >> 1) ? 8 : 0);
          const int n = nt * 8 + 2 * t + (e & 1);
          if (k < K && v != 0.f) atomicAdd(dW + k * NOUT + n, v);
        }
  }
}

}  // namespace stem

bool scn_stem_tc_shape_ok(int K, int n_in, int n_out) { return n_in == 1 && n_out == stem::NOUT && K >= 1 && K <= 16 * stem::MAXKT; }

// x: fp32 or bf16 [n_in_rows, 1]; W: fp32 [K][1][32]; out: bf16 or fp32 [n_rows, 32]
int scn_stem_tc_forward(const void* x, int x_dtype, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, const float* W,
                        const float* bias, void* out, int out_dtype, cudaStream_t s) {
  const int64_t tiles = (n_rows + 15) / 16;
  int64_t g = (tiles + 7) / 8;
  if (g > (int64_t)kNumSMs * 3) g = (int64_t)kNumSMs * 3;
  if (g < 1) g = 1;
  auto launch = [&](auto kern, auto xp, auto op) -> int {
    SCN_CUDA(scn_launch_pdl(kern, dim3((unsigned)g), dim3(256), 0, s, xp, nbr, K, n_rows, n_pad, W, bias, op));
    SCN_LAUNCH_CHECK();
    return SCN_OK;
  };
  const float* xf = (const float*)x;
  const __nv_bfloat16* xb = (const __nv_bfloat16*)x;
  if (out_dtype == SCN_BF16) {
    if (x_dtype == SCN_F32) return launch(stem::k_stem_fwd<float, __nv_bfloat16>, xf, (__nv_bfloat16*)out);
    if (x_dtype == SCN_BF16) return launch(stem::k_stem_fwd<__nv_bfloat16, __nv_bfloat16>, xb, (__nv_bfloat16*)out);
  } else if (out_dtype == SCN_F32) {
    if (x_dtype == SCN_F32) return launch(stem::k_stem_fwd<float, float>, xf, (float*)out);
  }
  return SCN_ERR_ARG;
}

// dW: fp32 [K][1][32], accumulated into; dout: bf16, or fp32 with fp32 x
int scn_stem_tc_wgrad(const void* x, int x_dtype, const void* dout, int dout_dtype, const int32_t* nbr, int K, int64_t n_rows,
                      int64_t n_pad, float* dW, cudaStream_t s) {
  const int64_t tiles = (n_rows + 15) / 16;
  int64_t g = (tiles + 1) / 2;
  if (g > (int64_t)kNumSMs * 2) g = (int64_t)kNumSMs * 2;
  if (g < 1) g = 1;
  auto launch = [&](auto kern, auto xp, auto dp) -> int {
    SCN_CUDA(scn_launch_pdl(kern, dim3((unsigned)g), dim3(256), 0, s, xp, dp, nbr, K, n_rows, n_pad, dW));
    SCN_LAUNCH_CHECK();
    return SCN_OK;
  };
  const float* xf = (const float*)x;
  const __nv_bfloat16* db = (const __nv_bfloat16*)dout;
  if (dout_dtype == SCN_BF16) {
    if (x_dtype == SCN_F32) return launch(stem::k_stem_wgrad<float, __nv_bfloat16>, xf, db);
    if (x_dtype == SCN_BF16) return launch(stem::k_stem_wgrad<__nv_bfloat16, __nv_bfloat16>, (const __nv_bfloat16*)x, db);
  } else if (dout_dtype == SCN_F32) {
    if (x_dtype == SCN_F32) return launch(stem::k_stem_wgrad<float, float>, xf, (const float*)dout);
  }
  return SCN_ERR_ARG;
}
