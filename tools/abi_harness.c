/*
 * abi_harness.c -- a caller of libscn_b200.so that is NOT PyTorch: plain C99 + the CUDA runtime.
 *
 * It walks the same sequence SparseConvNet's InputLayer -> SubmanifoldConvolution -> AveragePooling make
 * through the C ABI (include/scn_b200.h) on a small seeded event and checks every result against loops
 * written here: InputLayer row numbering (first appearance, duplicates summed), the 3x3x3 submanifold
 * convolution on the exact-fp32 path (3 -> 5 planes) and on the tcgen05 path (32 -> 32 planes, bf16
 * features; the check rounds its operands to bf16 like the kernel's inputs), and 2x2x2 average pooling.
 *
 * Build (tests/test_abi.py does this on the CPU box; running needs a B200):
 *   gcc -std=c99 -O2 -Iinclude -I/usr/local/cuda/include tools/abi_harness.c \
 *       -Lsparseeventid_b200/lib -lscn_b200 -L/usr/local/cuda/lib64 -lcudart -lm -o abi_harness
 *   LD_LIBRARY_PATH=sparseeventid_b200/lib ./abi_harness
 * Exit status 0 = every check passed.  Also a convenient single-process target for `ncu`.
 */
#include <cuda_runtime_api.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "scn_b200.h"

#define CK(call)                                                                                  \
  do {                                                                                            \
    int rc__ = (int)(call);                                                                       \
    if (rc__ != 0) {                                                                              \
      fprintf(stderr, "%s:%d: %s -> %d\n", __FILE__, __LINE__, #call, rc__);                      \
      exit(2);                                                                                    \
    }                                                                                             \
  } while (0)

static uint32_t rng_state = 12345u;
static uint32_t rng(void) {
  rng_state = rng_state * 1664525u + 1013904223u;
  return rng_state >> 8;
}
static float rng_unit(void) { return (float)(rng() % 20001) / 10000.0f - 1.0f; }

/* bf16 round-to-nearest-even of an fp32 value, returned as fp32 (what the tensor-core path feeds the MMA) */
static float bf16_round(float v) {
  uint32_t u;
  memcpy(&u, &v, 4);
  u += 0x7FFFu + ((u >> 16) & 1u);
  u &= 0xFFFF0000u;
  memcpy(&v, &u, 4);
  return v;
}

static void* dmalloc(size_t bytes) {
  void* p = NULL;
  CK(cudaMalloc(&p, bytes ? bytes : 1));
  return p;
}
static void h2d(void* d, const void* h, size_t bytes) { CK(cudaMemcpy(d, h, bytes, cudaMemcpyHostToDevice)); }
static void d2h(void* h, const void* d, size_t bytes) { CK(cudaMemcpy(h, d, bytes, cudaMemcpyDeviceToHost)); }

static int find_row(const int32_t* act, int n_act, int x, int y, int z, int b) {
  for (int r = 0; r < n_act; ++r)
    if (act[4 * r] == x && act[4 * r + 1] == y && act[4 * r + 2] == z && act[4 * r + 3] == b) return r;
  return -1;
}

/* out[o] = bias + sum_k in[row(site(o) + d_k)] . W[k], offsets row-major over [-1,1]^3, last axis fastest */
static void conv_check(const int32_t* act, int n_act, const float* in, int cin, int cout, const float* W,
                       const float* bias, int round_operands, double* out) {
  for (int o = 0; o < n_act; ++o) {
    for (int c = 0; c < cout; ++c) out[(size_t)o * cout + c] = bias[c];
    int k = 0;
    for (int dx = -1; dx <= 1; ++dx)
      for (int dy = -1; dy <= 1; ++dy)
        for (int dz = -1; dz <= 1; ++dz, ++k) {
          int i = find_row(act, n_act, act[4 * o] + dx, act[4 * o + 1] + dy, act[4 * o + 2] + dz, act[4 * o + 3]);
          if (i < 0) continue;
          for (int a = 0; a < cin; ++a) {
            float xv = in[(size_t)i * cin + a];
            if (round_operands) xv = bf16_round(xv);
            for (int c = 0; c < cout; ++c) {
              float wv = W[((size_t)k * cin + a) * cout + c];
              if (round_operands) wv = bf16_round(wv);
              out[(size_t)o * cout + c] += (double)xv * (double)wv;
            }
          }
        }
  }
}

static double rel_l2(const float* got, const double* want, size_t n) {
  double num = 0, den = 0;
  for (size_t i = 0; i < n; ++i) {
    num += (got[i] - want[i]) * (got[i] - want[i]);
    den += want[i] * want[i];
  }
  return sqrt(num / (den > 0 ? den : 1));
}

/* one submanifold convolution through the C ABI; features converted to feat_dtype on the device */
static double run_conv(const float* x_dev_f32, const int32_t* nbr_dev, int64_t n_act, int64_t n_pad, int cin, int cout,
                       int precision, int feat_dtype, const float* W, const float* bias, const int32_t* act,
                       const float* x_host) {
  const int K = 27;
  size_t esz = feat_dtype == SCN_BF16 ? 2 : 4;
  float* W_dev = (float*)dmalloc((size_t)K * cin * cout * 4);
  float* b_dev = (float*)dmalloc((size_t)cout * 4);
  h2d(W_dev, W, (size_t)K * cin * cout * 4);
  h2d(b_dev, bias, (size_t)cout * 4);
  void* wimg = dmalloc(scn_conv_prep_bytes(K, cin, cout, precision, feat_dtype));
  CK(scn_conv_prep_weights(W_dev, K, cin, cout, 0, 0, precision, feat_dtype, wimg, NULL));
  void* x_dev = dmalloc((size_t)n_act * cin * esz);
  void* y_dev = dmalloc((size_t)n_act * cout * esz);
  float* y32_dev = (float*)dmalloc((size_t)n_act * cout * 4);
  /* rows == NULL: plain element-type conversion of an [n, C] matrix */
  CK(scn_rows_gather(x_dev_f32, SCN_F32, NULL, n_act, cin, x_dev, feat_dtype, NULL));
  CK(scn_conv_forward(x_dev, feat_dtype, n_act, nbr_dev, K, n_act, n_pad, cin, cout, wimg, b_dev, precision, y_dev,
                      feat_dtype, NULL));
  CK(scn_rows_gather(y_dev, feat_dtype, NULL, n_act, cout, y32_dev, SCN_F32, NULL));
  CK(cudaDeviceSynchronize());
  float* y = (float*)malloc((size_t)n_act * cout * 4);
  double* want = (double*)malloc((size_t)n_act * cout * 8);
  d2h(y, y32_dev, (size_t)n_act * cout * 4);
  conv_check(act, (int)n_act, x_host, cin, cout, W, bias, precision == SCN_PREC_BF16, want);
  double e = rel_l2(y, want, (size_t)n_act * cout);
  printf("  conv 3x3x3 %d->%d path %d (%s features): rel L2 err %.3e\n", cin, cout,
         scn_conv_path(K, cin, cout, precision, feat_dtype), feat_dtype == SCN_BF16 ? "bf16" : "fp32", e);
  free(y);
  free(want);
  cudaFree(W_dev); cudaFree(b_dev); cudaFree(wimg); cudaFree(x_dev); cudaFree(y_dev); cudaFree(y32_dev);
  return e;
}

int main(void) {
  enum { N_IN = 600, GRID = 24, BATCH = 2, CMAX = 32 };
  int failures = 0;
  printf("%s, %llu launches so far\n", scn_version(), (unsigned long long)scn_launch_count());

  /* ---- a seeded event: two random walks (tracks) per sample, revisits = duplicate input rows ---- */
  static int32_t coords[N_IN * 4];
  static float feats[N_IN * CMAX];
  int p[3] = {GRID / 2, GRID / 2, GRID / 2};
  for (int i = 0; i < N_IN; ++i) {
    int b = i * BATCH / N_IN;
    if (i % (N_IN / (2 * BATCH)) == 0) p[0] = p[1] = p[2] = GRID / 2;
    int axis = (int)(rng() % 3);
    p[axis] += (rng() & 1) ? 1 : -1;
    if (p[axis] < 0) p[axis] = 0;
    if (p[axis] >= GRID) p[axis] = GRID - 1;
    coords[4 * i] = p[0]; coords[4 * i + 1] = p[1]; coords[4 * i + 2] = p[2]; coords[4 * i + 3] = b;
    for (int c = 0; c < CMAX; ++c) feats[i * CMAX + c] = rng_unit();
  }

  /* ---- InputLayer: host restatement (first-appearance rows, duplicates summed) ---- */
  static int32_t act[N_IN * 4], row_want[N_IN];
  static float x_want[N_IN * CMAX];
  int n_act_want = 0;
  memset(x_want, 0, sizeof x_want);
  for (int i = 0; i < N_IN; ++i) {
    int r = find_row(act, n_act_want, coords[4 * i], coords[4 * i + 1], coords[4 * i + 2], coords[4 * i + 3]);
    if (r < 0) {
      r = n_act_want++;
      memcpy(act + 4 * r, coords + 4 * i, 16);
    }
    row_want[i] = r;
    for (int c = 0; c < CMAX; ++c) x_want[r * CMAX + c] += feats[i * CMAX + c];
  }

  /* ---- InputLayer through the C ABI ---- */
  int32_t* coords_dev = (int32_t*)dmalloc(sizeof coords);
  h2d(coords_dev, coords, sizeof coords);
  uint64_t* keys_in = (uint64_t*)dmalloc(N_IN * 8);
  CK(scn_pack_coords_checked(coords_dev, SCN_COORD_I32, N_IN, 4, 3, keys_in, NULL, NULL));
  int64_t cap = scn_hash_capacity(N_IN);
  uint64_t* tkeys = (uint64_t*)dmalloc((size_t)cap * 8);
  int32_t* tvals = (int32_t*)dmalloc((size_t)cap * 4);
  int32_t* row_dev = (int32_t*)dmalloc(N_IN * 4);
  uint64_t* keys_act = (uint64_t*)dmalloc(N_IN * 8);
  int32_t* n_act_dev = (int32_t*)dmalloc(4);
  size_t ws_bytes = scn_input_rules_workspace(N_IN);
  void* ws = dmalloc(ws_bytes);
  CK(scn_input_layer_rules(keys_in, N_IN, tkeys, tvals, cap, row_dev, keys_act, n_act_dev, ws, ws_bytes, NULL));
  int32_t n_act = 0;
  d2h(&n_act, n_act_dev, 4);
  static int32_t row_got[N_IN], act_got[N_IN * 4];
  d2h(row_got, row_dev, sizeof row_got);
  int32_t* act_dev = (int32_t*)dmalloc(N_IN * 16);
  CK(scn_unpack_keys(keys_act, n_act, act_dev, NULL));
  d2h(act_got, act_dev, (size_t)n_act * 16);
  int ok = n_act == n_act_want && memcmp(row_got, row_want, sizeof row_got) == 0 &&
           memcmp(act_got, act, (size_t)n_act * 16) == 0;
  printf("InputLayer rules: %d input rows -> %d active sites (want %d): %s\n", N_IN, n_act, n_act_want,
         ok ? "bit-exact" : "MISMATCH");
  failures += !ok;
  if (!ok) return 1;

  float* feats_dev = (float*)dmalloc(sizeof feats);
  h2d(feats_dev, feats, sizeof feats);
  float* x_dev = (float*)dmalloc((size_t)n_act * CMAX * 4);
  CK(scn_input_layer_forward(feats_dev, row_dev, N_IN, n_act, CMAX, 3, x_dev, SCN_F32, NULL, NULL));
  static float x_got[N_IN * CMAX];
  d2h(x_got, x_dev, (size_t)n_act * CMAX * 4);
  double worst = 0;
  for (int i = 0; i < n_act * CMAX; ++i) worst = fmax(worst, fabs((double)x_got[i] - x_want[i]));
  printf("InputLayer features (duplicates summed): max abs err %.3e\n", worst);
  failures += worst > 1e-5;

  /* ---- submanifold rulebook + convolutions ---- */
  int64_t n_pad = (n_act + 127) / 128 * 128;
  int32_t* nbr = (int32_t*)dmalloc((size_t)27 * n_pad * 4);
  CK(scn_subm_rulebook(keys_act, n_act, tkeys, tvals, cap, 3, 3, 3, nbr, n_pad, NULL));
  static float W[27 * CMAX * CMAX], bias[CMAX];
  for (size_t i = 0; i < sizeof W / 4; ++i) W[i] = 0.2f * rng_unit();
  for (int i = 0; i < CMAX; ++i) bias[i] = rng_unit();
  {
    /* exact fp32 path: first 3 feature planes -> 5 planes */
    static float x3[N_IN * 3];
    for (int r = 0; r < n_act; ++r)
      for (int c = 0; c < 3; ++c) x3[r * 3 + c] = x_want[r * CMAX + c];
    float* x3_dev = (float*)dmalloc((size_t)n_act * 3 * 4);
    h2d(x3_dev, x3, (size_t)n_act * 3 * 4);
    double e = run_conv(x3_dev, nbr, n_act, n_pad, 3, 5, SCN_PREC_FP32, SCN_F32, W, bias, act, x3);
    failures += !(e <= 1e-5);
    cudaFree(x3_dev);
  }
  {
    /* tensor-core path (tcgen05 + TMEM): 32 -> 32 planes, bf16 features */
    double e = run_conv(x_dev, nbr, n_act, n_pad, CMAX, CMAX, SCN_PREC_BF16, SCN_BF16, W, bias, act, x_want);
    failures += !(e <= 4e-3);          /* fp32 accumulate; the result itself is stored as bf16 (2^-9 relative) */
  }

  /* ---- AveragePooling 2x2x2: strided rulebook, tables, gather-sum ---- */
  {
    size_t sws_bytes = scn_strided_hash_workspace(n_act);
    void* sws = dmalloc(sws_bytes);
    int64_t ocap = scn_hash_capacity(n_act);
    uint64_t* otkeys = (uint64_t*)dmalloc((size_t)ocap * 8);
    int32_t* otvals = (int32_t*)dmalloc((size_t)ocap * 4);
    uint64_t* keys_out = (uint64_t*)dmalloc((size_t)n_act * 8);
    int32_t* out_row = (int32_t*)dmalloc((size_t)n_act * 4);
    int32_t* off = (int32_t*)dmalloc((size_t)n_act * 4);
    int32_t* n_out_dev = (int32_t*)dmalloc(4);
    CK(scn_strided_rulebook_hash(keys_act, n_act, 2, 2, 2, otkeys, otvals, ocap, keys_out, out_row, off, n_out_dev, sws,
                                 sws_bytes, NULL));
    int32_t n_out = 0;
    d2h(&n_out, n_out_dev, 4);
    int64_t n_out_pad = (n_out + 127) / 128 * 128;
    int32_t* down = (int32_t*)dmalloc((size_t)8 * n_out_pad * 4);
    int32_t* up = (int32_t*)dmalloc((size_t)8 * n_pad * 4);
    CK(scn_strided_tables(out_row, off, n_act, 8, down, n_out_pad, up, n_pad, NULL));
    float* y_dev = (float*)dmalloc((size_t)n_out * CMAX * 4);
    CK(scn_pool_rows(x_dev, SCN_F32, CMAX, down, 8, n_out, n_out_pad, CMAX, 1.0f / 8, y_dev, NULL));
    int32_t* oc_dev = (int32_t*)dmalloc((size_t)n_out * 16);
    CK(scn_unpack_keys(keys_out, n_out, oc_dev, NULL));
    int32_t* oc = (int32_t*)malloc((size_t)n_out * 16);
    float* y = (float*)malloc((size_t)n_out * CMAX * 4);
    d2h(oc, oc_dev, (size_t)n_out * 16);
    d2h(y, y_dev, (size_t)n_out * CMAX * 4);
    double bad = 0;
    int covered = 0;
    for (int q = 0; q < n_out; ++q)
      for (int c = 0; c < CMAX; ++c) {
        double s = 0;
        for (int r = 0; r < n_act; ++r)
          if (act[4 * r] / 2 == oc[4 * q] && act[4 * r + 1] / 2 == oc[4 * q + 1] && act[4 * r + 2] / 2 == oc[4 * q + 2] &&
              act[4 * r + 3] == oc[4 * q + 3]) {
            s += x_want[r * CMAX + c];
            covered += c == 0;
          }
        bad = fmax(bad, fabs(s / 8 - y[q * CMAX + c]));
      }
    printf("AveragePooling 2x2x2: %d -> %d sites, every input row pooled once: %s, max abs err %.3e\n", n_act, n_out,
           covered == n_act ? "yes" : "NO", bad);
    failures += covered != n_act || bad > 1e-5;
    free(oc);
    free(y);
  }
  CK(cudaDeviceSynchronize());
  printf("%llu kernels of libscn_b200 launched; %s\n", (unsigned long long)scn_launch_count(),
         failures ? "FAILED" : "all checks passed");
  return failures ? 1 : 0;
}
