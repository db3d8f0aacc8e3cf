/*
 * scn_oracle_c.c -- plain-C restatement of the INTEGER part of SparseConvNet's algorithm for this path (row numbering,
 * submanifold and strided rulebooks) and an fp64 rulebook convolution.
 *
 * TEST INFRASTRUCTURE ONLY (tests/ and __graft_entry__.build() compile and load it; the product never does).
 * PARITY UNPINNED vs SparseConvNet itself, like oracle/scn_oracle.py (SCN is an un-vendored, un-pinned dependency of
 * the reference and absent from the image).  Its purpose is to be a SECOND, independently written implementation of
 * the same published semantics (SURVEY.md App. A), in another language and with another data structure (a chained
 * hash map here, sorted arrays + searchsorted in the Python oracle), so that the two oracles pin each other.
 *
 * Reference call sites whose behaviour is restated (relative to /root/reference):
 *   scn.InputLayer            src/networks/resnet.py:26-29,143       first-appearance row numbering, one counter per batch
 *   scn.SubmanifoldConvolution src/networks/sparse_building_blocks.py:29-34   rules[k] = {(row(p + d_k), row(p))}
 *   scn.Convolution (f == s)  src/networks/sparse_building_blocks.py:110-117  q = floor(p / s), k = rowmajor(p - q s)
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct { int64_t key; int32_t row; int32_t next; } Node;
typedef struct { int32_t* head; Node* nodes; int64_t cap; int64_t n; } Map;

static uint64_t mix(uint64_t k) { k ^= k >> 31; k *= 0x9E3779B97F4A7C15ull; k ^= k >> 29; return k; }
static int map_init(Map* m, int64_t n) {
  m->cap = 16; while (m->cap < 2 * n) m->cap <<= 1;
  m->head = (int32_t*)malloc(sizeof(int32_t) * (size_t)m->cap);
  m->nodes = (Node*)malloc(sizeof(Node) * (size_t)(n > 0 ? n : 1));
  m->n = 0;
  if (!m->head || !m->nodes) return -1;
  for (int64_t i = 0; i < m->cap; ++i) m->head[i] = -1;
  return 0;
}
static void map_free(Map* m) { free(m->head); free(m->nodes); }
static int32_t map_get(const Map* m, int64_t key) {
  for (int32_t i = m->head[mix((uint64_t)key) & (uint64_t)(m->cap - 1)]; i >= 0; i = m->nodes[i].next)
    if (m->nodes[i].key == key) return m->nodes[i].row;
  return -1;
}
static void map_put(Map* m, int64_t key, int32_t row) {
  uint64_t b = mix((uint64_t)key) & (uint64_t)(m->cap - 1);
  Node* nd = &m->nodes[m->n];
  nd->key = key; nd->row = row; nd->next = m->head[b];
  m->head[b] = (int32_t)m->n++;
}

/* (x0, x1, x2, batch) -> batch:16 | x0:16 | x1:16 | x2:16 ; lexicographic (batch, x0, x1, x2) == numeric order of the
 * UNSIGNED key (batch indices >= 32768 set the top bit) */
static uint64_t pack(const int64_t* c) {
  return ((uint64_t)c[3] << 48) | ((uint64_t)c[0] << 32) | ((uint64_t)c[1] << 16) | (uint64_t)c[2];
}

/* InputLayer: coords int64 [n][4] (batch LAST).  Writes row_of_input[n], active[n_active][4]; returns n_active. */
int64_t oc_input_rules(const int64_t* coords, int64_t n, int64_t* row_of_input, int64_t* active) {
  Map m;
  if (map_init(&m, n)) return -1;
  int64_t rows = 0;
  for (int64_t i = 0; i < n; ++i) {
    int64_t key = pack(coords + 4 * i);
    int32_t r = map_get(&m, key);
    if (r < 0) {                                  /* first appearance: next row number */
      r = (int32_t)rows;
      map_put(&m, key, r);
      memcpy(active + 4 * rows, coords + 4 * i, 4 * sizeof(int64_t));
      ++rows;
    }
    row_of_input[i] = r;
  }
  map_free(&m);
  return rows;
}

/* Submanifold rulebook of `n` UNIQUE active sites in row order.  Offsets enumerate the box row-major, last axis
 * fastest.  pair_in/pair_out: capacity K*n; offsets[K+1]: start of every offset's pairs (pairs ordered by out row). */
int oc_subm_rules(const int64_t* coords, int64_t n, int f0, int f1, int f2, int32_t* pair_in, int32_t* pair_out,
                  int64_t* offsets) {
  Map m;
  if (map_init(&m, n)) return -1;
  for (int64_t i = 0; i < n; ++i) map_put(&m, pack(coords + 4 * i), (int32_t)i);
  int64_t p = 0;
  int k = 0;
  for (int d0 = -(f0 / 2); d0 <= f0 / 2; ++d0)
    for (int d1 = -(f1 / 2); d1 <= f1 / 2; ++d1)
      for (int d2 = -(f2 / 2); d2 <= f2 / 2; ++d2, ++k) {
        offsets[k] = p;
        for (int64_t i = 0; i < n; ++i) {
          int64_t q[4] = {coords[4 * i] + d0, coords[4 * i + 1] + d1, coords[4 * i + 2] + d2, coords[4 * i + 3]};
          if (q[0] < 0 || q[1] < 0 || q[2] < 0 || q[0] > 65535 || q[1] > 65535 || q[2] > 65535) continue;
          int32_t j = map_get(&m, pack(q));
          if (j >= 0) { pair_in[p] = j; pair_out[p] = (int32_t)i; ++p; }
        }
      }
  offsets[k] = p;
  map_free(&m);
  return 0;
}

static int cmp_u64(const void* a, const void* b) {
  uint64_t x = *(const uint64_t*)a, y = *(const uint64_t*)b;
  return x < y ? -1 : (x > y ? 1 : 0);
}

/* Strided convolution with filter == stride: every input site p has exactly one output q = floor(p / s) and offset
 * k = rowmajor(p - q s).  Output rows are numbered by ascending (batch, x0, x1, x2).
 * Writes out_coords[n_out][4] (capacity n), out_row_of_in[n], off_of_in[n]; returns n_out. */
int64_t oc_strided_rules(const int64_t* coords, int64_t n, int s0, int s1, int s2, int64_t* out_coords,
                         int32_t* out_row_of_in, int32_t* off_of_in) {
  uint64_t* keys = (uint64_t*)calloc((size_t)(n > 0 ? n : 1), sizeof(uint64_t));
  if (!keys) return -1;
  const int s[3] = {s0, s1, s2};
  for (int64_t i = 0; i < n; ++i) {
    int64_t q[4];
    int k = 0;
    for (int a = 0; a < 3; ++a) {
      q[a] = coords[4 * i + a] / s[a];
      k = k * s[a] + (int)(coords[4 * i + a] - q[a] * s[a]);
    }
    q[3] = coords[4 * i + 3];
    keys[i] = pack(q);
    off_of_in[i] = k;
  }
  uint64_t* sorted = (uint64_t*)malloc(sizeof(uint64_t) * (size_t)(n > 0 ? n : 1));
  if (!sorted) { free(keys); return -1; }
  memcpy(sorted, keys, sizeof(uint64_t) * (size_t)n);
  qsort(sorted, (size_t)n, sizeof(uint64_t), cmp_u64);
  int64_t m = 0;
  for (int64_t i = 0; i < n; ++i)
    if (i == 0 || sorted[i] != sorted[i - 1]) sorted[m++] = sorted[i];
  for (int64_t r = 0; r < m; ++r) {
    out_coords[4 * r + 3] = (int64_t)(sorted[r] >> 48);
    out_coords[4 * r + 0] = (sorted[r] >> 32) & 0xFFFF;
    out_coords[4 * r + 1] = (sorted[r] >> 16) & 0xFFFF;
    out_coords[4 * r + 2] = sorted[r] & 0xFFFF;
  }
  for (int64_t i = 0; i < n; ++i) {               /* binary search of the input's coarse key */
    int64_t lo = 0, hi = m - 1;
    while (lo < hi) { int64_t mid = (lo + hi) / 2; if (sorted[mid] < keys[i]) lo = mid + 1; else hi = mid; }
    out_row_of_in[i] = (int32_t)lo;
  }
  free(keys); free(sorted);
  return m;
}

/* out[o][:] = bias + sum over pairs (i, o) of offset k:  x[i][:] . W[k]   (fp64; W [K][cin][cout]) */
void oc_conv_forward(const double* x, const double* W, const double* bias, const int32_t* pair_in,
                     const int32_t* pair_out, const int64_t* offsets, int K, int cin, int cout, int64_t n_out,
                     double* out) {
  for (int64_t o = 0; o < n_out; ++o)
    for (int c = 0; c < cout; ++c) out[o * cout + c] = bias ? bias[c] : 0.0;
  for (int k = 0; k < K; ++k)
    for (int64_t p = offsets[k]; p < offsets[k + 1]; ++p) {
      const double* xi = x + (int64_t)pair_in[p] * cin;
      double* oo = out + (int64_t)pair_out[p] * cout;
      const double* w = W + (int64_t)k * cin * cout;
      for (int a = 0; a < cin; ++a)
        for (int c = 0; c < cout; ++c) oo[c] += xi[a] * w[a * cout + c];
    }
}
