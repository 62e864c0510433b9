/*
 * sample_ext_oracle.c — CPU restatement of weighted and with-replacement neighbour sampling and of
 * the edge ids (ofspmm_sample_neighbors_ex, include/ofspmm.h).  TEST INFRASTRUCTURE ONLY:
 * tests/_sample_ext_oracle.py compiles it with gcc (-ffp-contract=off) into a temporary directory
 * and loads it; the product package never does.
 *
 * It follows the definitions, not the device algorithm: weighted, every eligible key of a row is
 * computed and the pairs (key, j) are sorted, the first k taken; with replacement, draw t takes
 * position mulhi(x(s, v, t), deg) for t = 0 .. k-1.  The keys come from the same plain-C header as
 * the device code's (of-spmm_b200/csrc/sample_key.h), so they agree bit for bit.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../../of-spmm_b200/csrc/sample_key.h"

double oracle_neglog(double u) { return sk_neglog(u); }

void oracle_neglog_array(const double* u, int64_t n, double* out) {
  for (int64_t i = 0; i < n; ++i) out[i] = sk_neglog(u[i]);
}

/* x(s, v, j) = mix(mix(s ^ v) + j) */
static uint64_t x_key(uint64_t seed, int64_t v, int64_t j) { return sk_mix64(sk_mix64(seed ^ (uint64_t)v) + (uint64_t)j); }

/* The weight bits widened exactly to fp64: pbytes 4 = fp32, 2 = bf16 (the high half of an fp32). */
static double widen(const void* p, int pbytes, int64_t e) {
  uint32_t b;
  if (pbytes == 4) {
    memcpy(&b, (const char*)p + e * 4, 4);
  } else {
    uint16_t h;
    memcpy(&h, (const char*)p + e * 2, 2);
    b = (uint32_t)h << 16;
  }
  float f;
  memcpy(&f, &b, 4);
  return (double)f;
}

uint64_t oracle_weighted_key(uint64_t seed, int64_t v, int64_t j, double w) {
  return sk_weighted_key(x_key(seed, v, j), w);
}

typedef struct { uint64_t key; int64_t j; } pair_t;

static int cmp_pair(const void* a, const void* b) {
  const pair_t* x = (const pair_t*)a;
  const pair_t* y = (const pair_t*)b;
  if (x->key != y->key) return x->key < y->key ? -1 : 1;
  return x->j < y->j ? -1 : (x->j > y->j);
}

static int cmp_i64(const void* a, const void* b) {
  const int64_t x = *(const int64_t*)a, y = *(const int64_t*)b;
  return x < y ? -1 : (x > y);
}

static int64_t count_sorted(const int64_t* a, int64_t n, int64_t x, int64_t* first) {
  int64_t lo = 0, hi = n;
  while (lo < hi) { const int64_t mid = (lo + hi) / 2; if (a[mid] < x) lo = mid + 1; else hi = mid; }
  *first = lo;
  int64_t e = lo;
  while (e < n && a[e] == x) ++e;
  return e - lo;
}

static uint64_t mulhi64(uint64_t a, uint64_t b) { return (uint64_t)(((unsigned __int128)a * b) >> 64); }

/* ofspmm_sample_neighbors_ex restated literally for a square A of `rows` rows, given the
 * destinations' rows only: the entries of row dst[i] are seg_col / seg_val / seg_prob at
 * [seg_off[i], seg_off[i+1]), and entry j of that row is entry seg_base[i] + j of A (its edge id).
 * vbytes: bytes per value (0: pattern); pbytes: bytes per weight (0: no prob, 2: bf16, 4: fp32);
 * replace: draws with replacement (pbytes must be 0).  The caller sizes blk_col / blk_val / blk_eid
 * for the sum of k and src_nodes for num_dst + that sum.  counts as in the header. */
void oracle_sample_neighbors_ex(int64_t rows, const int64_t* dst, int64_t num_dst, const int64_t* seg_off,
                                const int64_t* seg_base, const int64_t* seg_col, const void* seg_val, int vbytes,
                                const void* seg_prob, int pbytes, int replace, int64_t fanout, uint64_t seed,
                                int64_t* blk_crow, int64_t* blk_col, void* blk_val, int64_t* blk_eid,
                                int64_t* src_nodes, int64_t* counts) {
  int64_t* sdst = (int64_t*)malloc(sizeof(int64_t) * (size_t)(num_dst > 0 ? num_dst : 1));
  memcpy(sdst, dst, sizeof(int64_t) * (size_t)num_dst);
  qsort(sdst, (size_t)num_dst, sizeof(int64_t), cmp_i64);
  int64_t nnz = 0, invalid = 0, first = 0;
  blk_crow[0] = 0;
  for (int64_t i = 0; i < num_dst; ++i) {
    const int64_t v = dst[i];
    if (v < 0 || v >= rows || count_sorted(sdst, num_dst, v, &first) != 1) {
      ++invalid;
      blk_crow[i + 1] = nnz;
      continue;
    }
    const int64_t b = seg_off[i], deg = seg_off[i + 1] - b;
    /* the positions taken, in the order the row holds them */
    int64_t* take = NULL;
    int64_t ntake = 0;
    if (replace && fanout != -1) {
      const int64_t k = deg > 0 ? fanout : 0;
      take = (int64_t*)malloc(sizeof(int64_t) * (size_t)(k > 0 ? k : 1));
      for (int64_t t = 0; t < k; ++t) take[ntake++] = (int64_t)mulhi64(x_key(seed, v, t), (uint64_t)deg);
    } else {
      pair_t* pairs = (pair_t*)malloc(sizeof(pair_t) * (size_t)(deg > 0 ? deg : 1));
      int64_t npos = 0;
      for (int64_t j = 0; j < deg; ++j) {
        if (pbytes) {
          const double w = widen(seg_prob, pbytes, b + j);
          if (!sk_eligible(w)) continue;
          pairs[npos].key = sk_weighted_key(x_key(seed, v, j), w);
        } else {
          pairs[npos].key = x_key(seed, v, j);
        }
        pairs[npos++].j = j;
      }
      const int64_t k = fanout == -1 ? npos : (npos < fanout ? npos : fanout);
      qsort(pairs, (size_t)npos, sizeof(pair_t), cmp_pair);
      char* chosen = (char*)calloc((size_t)(deg > 0 ? deg : 1), 1);
      for (int64_t t = 0; t < k; ++t) chosen[pairs[t].j] = 1;
      take = (int64_t*)malloc(sizeof(int64_t) * (size_t)(k > 0 ? k : 1));
      for (int64_t j = 0; j < deg; ++j)
        if (chosen[j]) take[ntake++] = j;
      free(chosen);
      free(pairs);
    }
    for (int64_t t = 0; t < ntake; ++t) {
      const int64_t j = take[t], c = seg_col[b + j];
      if (c < 0 || c >= rows) continue;   /* columns outside [0, cols) are dropped */
      blk_col[nnz] = c;
      blk_eid[nnz] = seg_base[i] + j;
      if (vbytes) memcpy((char*)blk_val + nnz * vbytes, (const char*)seg_val + (b + j) * vbytes, (size_t)vbytes);
      ++nnz;
    }
    free(take);
    blk_crow[i + 1] = nnz;
  }
  /* src_nodes = dst, then the distinct sampled ids that are not destinations, ascending */
  int64_t* ids = (int64_t*)malloc(sizeof(int64_t) * (size_t)(nnz > 0 ? nnz : 1));
  memcpy(ids, blk_col, sizeof(int64_t) * (size_t)nnz);
  qsort(ids, (size_t)nnz, sizeof(int64_t), cmp_i64);
  int64_t tail = 0;
  for (int64_t p = 0; p < nnz; ++p) {
    if (p > 0 && ids[p] == ids[p - 1]) continue;
    if (count_sorted(sdst, num_dst, ids[p], &first) > 0) continue;
    ids[tail++] = ids[p];
  }
  for (int64_t i = 0; i < num_dst; ++i) src_nodes[i] = dst[i];
  for (int64_t t = 0; t < tail; ++t) src_nodes[num_dst + t] = ids[t];
  /* local ids: position in dst, else num_dst + rank among the new ids */
  pair_t* where = (pair_t*)malloc(sizeof(pair_t) * (size_t)(num_dst > 0 ? num_dst : 1));
  for (int64_t i = 0; i < num_dst; ++i) { where[i].key = (uint64_t)dst[i]; where[i].j = i; }
  qsort(where, (size_t)num_dst, sizeof(pair_t), cmp_pair);
  for (int64_t p = 0; p < nnz; ++p) {
    const uint64_t c = (uint64_t)blk_col[p];
    int64_t lo = 0, hi = num_dst;
    while (lo < hi) { const int64_t mid = (lo + hi) / 2; if (where[mid].key < c) lo = mid + 1; else hi = mid; }
    if (lo < num_dst && where[lo].key == c) {
      blk_col[p] = where[lo].j;
    } else {
      count_sorted(ids, tail, (int64_t)c, &first);
      blk_col[p] = num_dst + first;
    }
  }
  free(where);
  counts[0] = nnz;
  counts[1] = num_dst + tail;
  counts[2] = invalid;
  free(ids);
  free(sdst);
}
