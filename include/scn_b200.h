/*
 * scn_b200.h -- C ABI of libscn_b200.so: the B200-native (sm_100a) replacement for the native
 * layer of SparseConvNet (`sparseconvnet.SCN`, a pybind11 module over C++ Metadata/sparsehash
 * rulebooks and CPU/CUDA kernels) that the reference reaches through every `scn.*` module.
 *
 * Plain pointers and sizes only; no torch types.  All pointers are DEVICE pointers unless the
 * name ends in `_host`.  Every entry point is stream-ordered on `stream` (a cudaStream_t passed
 * as void*), never synchronises the device unless stated, never throws, and returns 0 on
 * success, a positive cudaError_t value on a CUDA failure or a negative SCN_ERR_* code on a bad
 * argument.
 *
 * Reference interfaces replaced (paths relative to the reference repository; SCN symbols are the
 * upstream names the reference's call sites resolve to, SURVEY.md 2.2/2.3/8b):
 *   Metadata<D>/SparseGrid + InputLayer_updateOutput   <- scn.InputLayer   src/networks/resnet.py:26-29,40-43,143
 *   SubmanifoldConvolution_SgToRules / _updateOutput /
 *     _backward                                         <- scn.SubmanifoldConvolution
 *                                                          src/networks/sparse_building_blocks.py:29-34
 *                                                          src/networks/resnet.py:30-36,44-50,105-110
 *   Convolution_InputSgsToRulesAndOutputSgs /
 *     Convolution_updateOutput / _backward              <- scn.Convolution  src/networks/sparse_building_blocks.py:110-117
 *   Deconvolution_updateOutput / _backward              <- scn.Deconvolution src/networks/sparse_building_blocks.py:207-213
 *   BatchNormalization_updateOutput / _backward         <- scn.BatchNormalization(+ReLU/LeakyReLU)
 *                                                          src/networks/sparse_building_blocks.py:39,122
 *                                                          src/networks/torch/sparseresnet.py:28-29
 *   LeakyReLU_updateOutput / _updateGradInput           <- scn.LeakyReLU / scn.ReLU sparse_building_blocks.py:45,80,128
 *   AddTable                                            <- scn.AddTable     sparse_building_blocks.py:82,96
 *   SparseToDense_updateOutput / _updateGradInput       <- scn.SparseToDense src/networks/resnet.py:123-125
 *   OutputLayer_updateOutput / _updateGradInput         <- scn.OutputLayer  (named by the north star; no call site)
 *   AveragePooling_updateOutput / _updateGradInput      <- scn.AveragePooling sparse_building_blocks.py:150-154
 */
#ifndef SCN_B200_H
#define SCN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCN_OK 0
#define SCN_ERR_ARG (-1)          /* bad size / null pointer / unsupported combination */
#define SCN_ERR_UNSUPPORTED (-2)  /* shape outside what the kernels implement */
#define SCN_ERR_WORKSPACE (-3)    /* workspace too small */

/* element types of feature matrices */
#define SCN_F32 0
#define SCN_BF16 1
/* element types accepted for coordinate input */
#define SCN_COORD_I64 0
#define SCN_COORD_I32 1
#define SCN_COORD_F32 2
#define SCN_COORD_F64 3

/* Library version / build info: "scn_b200 <ver> sm_100a". */
const char* scn_version(void);
/* Number of kernels of this library launched by this process so far (bench.py's gpu_launches). */
uint64_t scn_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Coordinate hash (replaces google::dense_hash_map<Point<D>,Int> inside SCN's Metadata).
 * A site is one packed 64-bit key  (batch:16 | x0:16 | x1:16 | x2:16); missing trailing axes
 * (dimension < 3) are 0.  The table is open addressing over buckets of 8 slots probed
 * cooperatively by 8 lanes; `capacity` is a power of two >= 2*n (scn_hash_capacity).
 * ------------------------------------------------------------------------------------------ */
int64_t scn_hash_capacity(int64_t n);

/* coords: [n, ncols] row-major of `coord_dtype`; ncols == dimension+1 (batch index LAST, as
 * produced by src/io/data_transforms.py:43-46,242) or ncols == dimension (single sample).
 * info: int32[4] on the device (zeroed by the caller), or NULL for no range check; info[1] |= 1 when a coordinate
 * is outside [0, 65535] or a batch index outside [0, 65534] (two sites would alias in the 16-bit key fields; the
 * host side raises), info[2] = max batch index seen (SCN: batch size = max(argument, max index + 1)).  info[0] and
 * info[3] are free for the caller (the InputLayer host code has scn_input_layer_rules write n_active to info[0] so
 * that one read-back returns all three). */
int scn_pack_coords_checked(const void* coords, int coord_dtype, int64_t n, int ncols, int dimension,
                            uint64_t* keys, int32_t* info, void* stream);
/* keys -> int32 [n, 4] rows (x0, x1, x2, batch): SparseConvNetTensor.get_spatial_locations(). */
int scn_unpack_keys(const uint64_t* keys, int64_t n, int32_t* coords4, void* stream);

/* Clears the table and inserts n UNIQUE keys with value = row index. */
int scn_hash_build(const uint64_t* keys, int64_t n, uint64_t* table_keys, int32_t* table_vals,
                   int64_t capacity, void* stream);
/* out[i] = row of query key i, or -1. */
int scn_hash_lookup(const uint64_t* queries, int64_t n, const uint64_t* table_keys,
                    const int32_t* table_vals, int64_t capacity, int32_t* out, void* stream);

/* InputLayer rules (SCN InputLayer modes 0-4 share them): de-duplicates keys_in, numbers the
 * active sites in FIRST-APPEARANCE order with one counter over the whole batch, fills the table
 * (key -> row), keys_out[row], row_of_input[i]; *n_active_dev receives the number of rows.
 * workspace: scn_input_rules_workspace(n) bytes. */
size_t scn_input_rules_workspace(int64_t n);
int scn_input_layer_rules(const uint64_t* keys_in, int64_t n, uint64_t* table_keys,
                          int32_t* table_vals, int64_t capacity, int32_t* row_of_input,
                          uint64_t* keys_out, int32_t* n_active_dev, void* workspace,
                          size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Rulebooks.  The device-resident form is a NEIGHBOUR TABLE  nbr[K][n_pad] (int32, -1 = none):
 * nbr[k][o] is the input row that reaches output row o through kernel offset k.  The SCN form
 * (per offset, a list of (in,out) pairs) is derived from it by scn_rulebook_pairs and is what
 * the parity tests compare, order-normalised, with the oracle.  n_pad = n rounded up to 128.
 * ------------------------------------------------------------------------------------------ */
/* Submanifold: offsets enumerate the box [-f/2,+f/2] row-major, last axis fastest;
 * nbr[k][o] = row(site(o) + d_k).  Only (K-1)/2 offsets are probed; the rest follow from the
 * mirror symmetry (i,o) in rules[k] <=> (o,i) in rules[K-1-k]. */
int scn_subm_rulebook(const uint64_t* keys, int64_t n, const uint64_t* table_keys,
                      const int32_t* table_vals, int64_t capacity, int f0, int f1, int f2,
                      int32_t* nbr, int64_t n_pad, void* stream);

/* Strided convolution with filter == stride (every use in the reference): output site
 * q = floor(p / s), offset k = rowmajor(p mod s).  Output rows are numbered in FIRST-APPEARANCE
 * order over the input rows (SparseConvNet creates output rows on first touch).
 * Writes keys_out[0..n_out) (in that order), out_row_of_in[n], off_of_in[n], *n_out_dev, and
 * table_keys / table_vals (capacity >= scn_hash_capacity(n)) receive the coarse level's hash table.
 * workspace: scn_strided_hash_workspace(n) bytes. */
size_t scn_strided_hash_workspace(int64_t n);
int scn_strided_rulebook_hash(const uint64_t* keys_in, int64_t n, int s0, int s1, int s2,
                              uint64_t* table_keys, int32_t* table_vals, int64_t capacity,
                              uint64_t* keys_out, int32_t* out_row_of_in, int32_t* off_of_in,
                              int32_t* n_out_dev, void* workspace, size_t workspace_bytes, void* stream);
/* Neighbour tables of a strided rulebook: down[k][q] = input row with offset k under output q
 * (K x n_out_pad, used by Convolution fwd / Deconvolution dgrad) and up[k][p] = output row of
 * input p if its offset is k (K x n_in_pad, used by Convolution dgrad / Deconvolution fwd). */
int scn_strided_tables(const int32_t* out_row_of_in, const int32_t* off_of_in, int64_t n_in,
                       int K, int32_t* nbr_down, int64_t n_out_pad, int32_t* nbr_up,
                       int64_t n_in_pad, void* stream);

/* SCN-format rulebook from a neighbour table: pairs sorted by (k, out row).
 * scn_rulebook_count writes counts_dev[K]; after reading them the caller allocates P = sum
 * entries and calls scn_rulebook_pairs, which writes pair_in[P], pair_out[P], offsets_dev[K+1]. */
size_t scn_rulebook_workspace(int K, int64_t n_pad);
int scn_rulebook_count(const int32_t* nbr, int K, int64_t n, int64_t n_pad, int32_t* counts_dev,
                       void* stream);
int scn_rulebook_pairs(const int32_t* nbr, int K, int64_t n, int64_t n_pad, int32_t* pair_in,
                       int32_t* pair_out, int32_t* offsets_dev, void* workspace,
                       size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Convolution arithmetic.  One output-stationary gather-GEMM covers every forward and dgrad:
 *     out[o, :] = bias + sum_k  in[nbr[k][o], :] . B_k          (rows with nbr < 0 contribute 0)
 *   SubmanifoldConvolution fwd : nbr = subm table,  B_k = W[k]
 *   SubmanifoldConvolution dgrad: same table,       B_k = W[K-1-k]^T   (mirror symmetry)
 *   Convolution fwd / Deconvolution dgrad: nbr = down table, B_k = W[k] / W[k]^T
 *   Convolution dgrad / Deconvolution fwd: nbr = up table,   B_k = W[k]^T / W[k]
 * and one pair-reduction covers every wgrad:
 *     dW[k] += sum_o in[nbr[k][o], :]^T . dout[o, :]
 * `precision`: SCN_PREC_BF16 = bf16 operands on tensor cores, fp32 accumulate (features may be
 * stored fp32 or bf16); SCN_PREC_FP32 = exact fp32 FMA path (fp32 features only); SCN_PREC_TF32 =
 * fp32 features, TF32 operands on the tcgen05 tensor cores (10-bit mantissa), fp32 accumulate; shapes
 * outside the tcgen05 kernels run the exact fp32 FMA path, the one-channel stem its hi/lo bf16 split.
 * ------------------------------------------------------------------------------------------ */
#define SCN_PREC_FP32 0
#define SCN_PREC_BF16 1
#define SCN_PREC_TF32 2

/* Re-lays the fp32 SCN weight W[K][Cin][Cout] for one of the uses above.
 *   transpose=0: B_k = W[k] (Cin x Cout);  transpose=1: B_k = W[src]^T with src = mirror ? K-1-k : k.
 * Output element type follows precision (fp32 or bf16); n_in/n_out below are B_k's own dims. */
int scn_conv_prep_weights(const float* W, int K, int Cin, int Cout, int transpose, int mirror,
                          int precision, int feat_dtype, void* out, void* stream);
/* Every weight image of a network in one launch (a trainer calls it once per step, then passes skip_prep = 1 to the
 * module entry points below).  descs: DEVICE array of n x 8 int64 {W pointer, image pointer, K, Cin, Cout,
 * transpose | mirror << 1, index of the image's first element in the concatenated index space, precision (an image
 * for SCN_PREC_TF32 holds TF32 values, any other value builds the bf16 image)}; total =
 * sum of K*Cin*Cout.  Only for images of the tcgen05 path (scn_conv_path == 2); an image whose n_in is not a multiple
 * of 64 must have been zero-filled once (its unused half rows are never written). */
int scn_conv_prep_weights_batched(const void* descs, int n, int64_t total, void* stream);
/* Which kernel family runs a (K, n_in, n_out) contraction for features of feat_dtype:
 *   0 exact fp32 FMA (B_k fp32 [k][c][n]);  1 mma.sync tensor cores (B_k bf16 [k][n][c]);
 *   2 tcgen05 tensor cores + TMEM (B_k as pre-swizzled 128-byte-row tiles: bf16, or TF32 for SCN_PREC_TF32 with
 *     fp32 features).
 * scn_conv_prep_bytes is the size of the buffer scn_conv_prep_weights fills for that path. */
int scn_conv_path(int K, int n_in, int n_out, int precision, int feat_dtype);
size_t scn_conv_prep_bytes(int K, int n_in, int n_out, int precision, int feat_dtype);

/* in: [n_in_rows, n_in] of in_dtype; out: [n_out_rows, n_out] of out_dtype (fully overwritten);
 * nbr: [K][n_pad]; Bprep: output of scn_conv_prep_weights; bias: fp32 [n_out] or NULL. */
int scn_conv_forward(const void* in, int in_dtype, int64_t n_in_rows, const int32_t* nbr, int K,
                     int64_t n_out_rows, int64_t n_pad, int n_in, int n_out, const void* Bprep,
                     const float* bias, int precision, void* out, int out_dtype, void* stream);

/* dW: fp32 [K][n_in][n_out], ACCUMULATED into (caller zeroes); `in` rows are gathered through
 * nbr (the SAME table the forward used), dout rows are the table's own rows [n_rows, n_out]. */
int scn_conv_wgrad(const void* in, int in_dtype, const void* dout, int dout_dtype,
                   const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int n_in, int n_out,
                   int precision, float* dW, void* stream);


/* dbias[c] = sum_rows dout[r][c]  (fp32 out, overwritten, or out[c] += ... when accumulate != 0:
 * gradient accumulated in place).  stats_ws: 2*C doubles of scratch. */
int scn_col_sum_acc(const void* x, int dtype, int64_t n, int C, double* stats_ws, float* out,
                    int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------
 * One call per convolution module forward / backward (the X_updateOutput / X_backward pairs of
 * SCN's SubmanifoldConvolution, Convolution and Deconvolution): weight re-layout, contraction(s)
 * and bias-gradient reduction on caller-owned workspaces.
 *   W: the module's fp32 parameter [K][Cin][Cout]; wimg / wimg_t: scn_conv_prep_bytes() bytes for
 *   (K,Cin,Cout) / (K,Cout,Cin); skip_prep != 0 when the workspace already holds the image of
 *   the current W.  Forward: out = bias + conv(x) through nbr.  Backward (each part optional,
 *   NULL skips it): dx through nbr_bwd with W^T (mirror: W[K-1-k]^T, submanifold), dW += x^T dout
 *   through nbr_fwd (zero_dW clears it first), dbias (+)= column sums of dout.  When those column
 *   sums are already known (dout_colsum: fp32 [Cout], e.g. from scn_bn_backward_colsum), dbias
 *   (+)= dout_colsum without another pass over dout; dout_colsum = NULL computes them (stats_ws:
 *   2*Cout doubles of scratch).
 * ------------------------------------------------------------------------------------------ */
int scn_conv_module_forward(const void* x, int x_dtype, int64_t n_in_rows, const int32_t* nbr,
                            int K, int64_t n_out_rows, int64_t n_pad, int Cin, int Cout,
                            const float* W, const float* bias, int precision, void* wimg,
                            int skip_prep, void* out, int out_dtype, void* stream);
int scn_conv_module_backward_colsum(const void* x, int x_dtype, int64_t n_in_rows, const void* dout,
                             int dout_dtype, int64_t n_out_rows, const int32_t* nbr_fwd,
                             int64_t n_pad_fwd, const int32_t* nbr_bwd, int64_t n_pad_bwd, int K,
                             int Cin, int Cout, const float* W, int mirror, int precision,
                             void* wimg_t, int skip_prep, void* dx, float* dW, int zero_dW,
                             float* dbias, int accumulate_dbias, const float* dout_colsum, double* stats_ws, void* stream);

/* ------------------------------------------------------------------------------------------
 * Bandwidth-bound layers.  Feature matrices are [n, C] row-major of `dtype`.
 * ------------------------------------------------------------------------------------------ */
/* BatchNormalization, SCN conventions (eps, inverted momentum, unbiased running variance):
 *   train: stats over the n rows; running = momentum*running + (1-momentum)*batch
 *   y = (x-mean)*invstd*gamma+beta;  out = y > 0 ? y : leakiness*y
 * save_mean/save_invstd: fp32 [C] (written in train mode, read by the backward).
 * stats_ws: 2*C doubles of scratch. */
int scn_bn_forward(const void* x, int dtype, int64_t n, int C, const float* gamma,
                   const float* beta, float* running_mean, float* running_var, int training,
                   float eps, float momentum, float leakiness, float* save_mean,
                   float* save_invstd, double* stats_ws, void* out, void* stream);
/* dx, dgamma[C], dbeta[C] (fp32; overwritten, or accumulated into when accumulate_params != 0).
 * `training` selects batch- or running-stat form.  dx_colsum (fp32 [C], or NULL to skip it) receives
 * the sum over the n rows of dx[:, c] as stored: when the BatchNormalization follows a convolution
 * with a bias (src/networks/sparse_building_blocks.py:29-39) that IS the convolution's bias gradient
 * (SCN: Convolution backward, d_bias = column sums of d_output), produced in the pass that writes dx
 * instead of by one more pass over it. */
int scn_bn_backward_colsum(const void* x, const void* dout, int dtype, int64_t n, int C,
                           const float* gamma, const float* beta, const float* save_mean,
                           const float* save_invstd, int training, float leakiness, double* stats_ws,
                           void* dx, float* dgamma, float* dbeta, int accumulate_params,
                           float* dx_colsum, void* stream);

int scn_leaky_forward(const void* x, int dtype, int64_t count, float leak, void* out, void* stream);
int scn_leaky_backward(const void* x, const void* dout, int dtype, int64_t count, float leak,
                       void* dx, void* stream);
/* out = a + b, optionally followed by leaky (leak == 1 -> plain AddTable). */
int scn_add_forward(const void* a, const void* b, int dtype, int64_t count, float leak, void* out,
                    void* stream);

/* InputLayer features: out[row_of_input[i], :] (+)= in[i, :]  (out zeroed inside; mode 4 divides
 * by the multiplicity), and its backward / OutputLayer forward: gather by row_of_input. */
int scn_input_layer_forward(const float* in, const int32_t* row_of_input, int64_t n_in,
                            int64_t n_active, int C, int mode, void* out, int out_dtype,
                            float* count_ws, void* stream);
int scn_rows_gather(const void* src, int dtype, const int32_t* rows, int64_t n_rows, int C,
                    void* out, int out_dtype, void* stream);
int scn_rows_scatter_add(const void* src, int dtype, const int32_t* rows, int64_t n_rows, int C,
                         float* out_f32, void* stream);

/* scn.AveragePooling rows (pool_size == pool_stride; reference call site
 * src/networks/sparse_building_blocks.py:150-154): out[r, :] = scale * sum over the k < K table
 * entries nbr[k * n_pad + r] >= 0 of x[that row, 0..C), fp32 accumulation in ascending k.  Forward:
 * nbr = the strided rule's [K][n_out_pad] table, scale = 1 / pool volume (SparseConvNet divides by
 * the pool volume, not by the number of active inputs).  Backward: the same call with the
 * transposed [K][n_in_pad] table on d(out).  ldx = row stride of x in elements (>= C), so that
 * nFeaturesToDrop can read a column window of a wider matrix; out is dense [n_rows, C]. */
int scn_pool_rows(const void* x, int dtype, int ldx, const int32_t* nbr, int K, int64_t n_rows,
                  int64_t n_pad, int C, float scale, void* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * larcv batch-filler array -> SCN input tuple on the device (replaces the host numpy transforms
 * larcvsparse_to_scnsparse_3d / _2d, src/io/data_transforms.py:21-49,198-252).
 * larcv: fp32 [B][P][V][ncol], last column = value, padding rows have value == pad_value (-999).
 * scn_larcv_count: counts[p*B + b] = live rows of (sample b, plane p).  The caller turns them into
 * exclusive offsets (plane-major order, which is the reference's row order) and allocates N rows.
 * scn_larcv_compact: order-preserving compaction; layout 0 (3-D): coords4 = (x, y, z, b);
 * layout 1 (2-D): coords4 = (plane, y, x, b); features[N] = value.
 * ------------------------------------------------------------------------------------------ */
int scn_larcv_count(const float* larcv, int B, int P, int V, int ncol, float pad_value,
                    int32_t* counts, void* stream);
int scn_larcv_compact(const float* larcv, int B, int P, int V, int ncol, float pad_value,
                      const int64_t* row_offsets, int layout, int32_t* coords4, float* features,
                      void* stream);

/* SparseToDense: dense[b][c][x0][x1][x2] (fp32, zero-filled inside) <- x[row][c]; backward gathers. */
int scn_sparse_to_dense_forward(const void* x, int dtype, const uint64_t* keys, int64_t n, int C,
                                int batch, int s0, int s1, int s2, float* dense, void* stream);
int scn_sparse_to_dense_backward(const float* ddense, const uint64_t* keys, int64_t n, int C,
                                 int batch, int s0, int s1, int s2, void* dx, int dtype,
                                 void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SCN_B200_H */
