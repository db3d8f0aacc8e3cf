// One C-ABI call per module forward / backward: the counterpart of SCN's X_updateOutput / X_backward entry points
// (SURVEY.md 8b).  The host side of the reference is single-threaded Python, so the number of boundary crossings,
// allocations and kernel launches per module decides how fast a step can be ENQUEUED; these wrappers fold
// "re-lay the weights, run the contraction(s), reduce the bias gradient" into one call on caller-owned workspaces.
// Reference call sites: src/networks/sparse_building_blocks.py:29-34,110-117,207-213.
#include "common.cuh"

extern "C" int scn_conv_module_forward(const void* x, int x_dtype, int64_t n_in_rows, const int32_t* nbr, int K,
                                       int64_t n_out_rows, int64_t n_pad, int Cin, int Cout, const float* W,
                                       const float* bias, int precision, void* wimg, int skip_prep, void* out,
                                       int out_dtype, void* stream) {
  if (!W || !wimg) return SCN_ERR_ARG;
  if (!skip_prep) {
    int rc = scn_conv_prep_weights(W, K, Cin, Cout, 0, 0, precision, out_dtype, wimg, stream);
    if (rc != SCN_OK) return rc;
  }
  return scn_conv_forward(x, x_dtype, n_in_rows, nbr, K, n_out_rows, n_pad, Cin, Cout, wimg, bias, precision, out,
                          out_dtype, stream);
}

// conv.cu
int scn_conv_wgrad_fold(const void* in, int in_dtype, const void* dout, int dout_dtype, const int32_t* nbr, int K,
                        int64_t n_rows, int64_t n_pad, int n_in, int n_out, int precision, float* dW, const float* colsum,
                        float* dbias, int accumulate_dbias, bool* bias_folded, cudaStream_t s);

namespace {
__global__ void k_bias_from_colsum(const float* __restrict__ colsum, float* dbias, int C, int accumulate) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) dbias[c] = (accumulate ? dbias[c] : 0.f) + colsum[c];
}
}  // namespace

extern "C" int scn_conv_module_backward_colsum(const void* x, int x_dtype, int64_t n_in_rows, const void* dout,
                                               int dout_dtype, int64_t n_out_rows, const int32_t* nbr_fwd,
                                               int64_t n_pad_fwd, const int32_t* nbr_bwd, int64_t n_pad_bwd, int K, int Cin,
                                               int Cout, const float* W, int mirror, int precision, void* wimg_t,
                                               int skip_prep, void* dx, float* dW, int zero_dW, float* dbias,
                                               int accumulate_dbias, const float* dout_colsum, double* stats_ws,
                                               void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (!W || !dout) return SCN_ERR_ARG;
  // the column sums of dout are known (scn_bn_backward_colsum): the bias gradient needs no pass over dout; the addition
  // rides on the weight gradient's reduction kernel when that runs, else on a C-thread kernel below
  const bool fold = dbias != nullptr && dout_colsum != nullptr;
  bool bias_folded = false;
  int rc = SCN_OK;
  if (dx) {                                   // dgrad: the same gather-GEMM on the transposed (mirrored) weights
    if (!wimg_t || !nbr_bwd) return SCN_ERR_ARG;
    if (!skip_prep) {
      rc = scn_conv_prep_weights(W, K, Cin, Cout, 1, mirror, precision, x_dtype, wimg_t, stream);
      if (rc != SCN_OK) return rc;
    }
    rc = scn_conv_forward(dout, dout_dtype, n_out_rows, nbr_bwd, K, n_in_rows, n_pad_bwd, Cout, Cin, wimg_t, nullptr,
                          precision, dx, x_dtype, stream);
    if (rc != SCN_OK) return rc;
  }
  if (dW) {
    if (!x || !nbr_fwd) return SCN_ERR_ARG;
    if (zero_dW) SCN_CUDA(cudaMemsetAsync(dW, 0, (size_t)K * Cin * Cout * sizeof(float), s));
    rc = scn_conv_wgrad_fold(x, x_dtype, dout, dout_dtype, nbr_fwd, K, n_out_rows, n_pad_fwd, Cin, Cout, precision, dW,
                             fold ? dout_colsum : nullptr, dbias, accumulate_dbias, &bias_folded, s);
    if (rc != SCN_OK) return rc;
  }
  if (fold) {
    if (!bias_folded) {                        // no reduction kernel ran (no dW wanted, or another wgrad path)
      k_bias_from_colsum<<<(Cout + 255) / 256, 256, 0, s>>>(dout_colsum, dbias, Cout, accumulate_dbias);
      SCN_LAUNCH_CHECK();
    }
  } else if (dbias) {
    if (!stats_ws) return SCN_ERR_ARG;
    rc = scn_col_sum_acc(dout, dout_dtype, n_out_rows, Cout, stats_ws, dbias, accumulate_dbias, stream);
    if (rc != SCN_OK) return rc;
  }
  return SCN_OK;
}
