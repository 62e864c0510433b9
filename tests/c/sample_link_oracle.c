/*
 * sample_link_oracle.c — CPU restatement of the link-prediction pieces of include/ofspmm.h: the row
 * selection of neighbour sampling with an exclusion list (OFSPMM_SAMPLE_EXCLUDE), negative sampling
 * and edge lookup.  TEST INFRASTRUCTURE ONLY: tests/_sample_link_oracle.py compiles it together
 * with sample_ext_oracle.c (whose weighted key it calls, so that neglog and the key are written
 * once) into a temporary directory; the product package never loads it.
 *
 * It follows the definitions, not the device algorithms: every eligible key of a row is computed
 * and the pairs (key, j) sorted; a draw with replacement maps its rank over the list of eligible
 * positions; a negative draw loops over its trials and tests membership by scanning the row.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../../of-spmm_b200/csrc/sample_key.h"

uint64_t oracle_weighted_key(uint64_t seed, int64_t v, int64_t j, double w); /* sample_ext_oracle.c */

static uint64_t x_key(uint64_t seed, int64_t v, int64_t j) { return sk_mix64(sk_mix64(seed ^ (uint64_t)v) + (uint64_t)j); }

static uint64_t mulhi64(uint64_t a, uint64_t b) { return (uint64_t)(((unsigned __int128)a * b) >> 64); }

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

typedef struct { uint64_t key; int64_t j; } lpair_t;

static int cmp_lpair(const void* a, const void* b) {
  const lpair_t* x = (const lpair_t*)a;
  const lpair_t* y = (const lpair_t*)b;
  if (x->key != y->key) return x->key < y->key ? -1 : 1;
  return x->j < y->j ? -1 : (x->j > y->j);
}

static int in_sorted(const int64_t* a, int64_t n, int64_t x) {
  int64_t lo = 0, hi = n;
  while (lo < hi) { const int64_t mid = (lo + hi) / 2; if (a[mid] < x) lo = mid + 1; else hi = mid; }
  return lo < n && a[lo] == x;
}

/* The positions (offsets j in the row, in the order the block holds them) that
 * ofspmm_sample_neighbors_ex takes from row v of `deg` entries starting at position `base` of A,
 * with the strictly ascending exclusion list excl[0, nexcl).  prob (pbytes 4 = fp32, 2 = bf16, 0 =
 * none) holds the row's weights; replace: draws with replacement.  take must hold deg entries
 * (replace: fanout).  Returns the number taken. */
int64_t oracle_take_row(int64_t v, int64_t base, int64_t deg, const void* prob, int pbytes, int replace,
                        int64_t fanout, uint64_t seed, const int64_t* excl, int64_t nexcl, int64_t* take) {
  int64_t* elig = (int64_t*)malloc(sizeof(int64_t) * (size_t)(deg > 0 ? deg : 1));
  int64_t ne = 0;
  for (int64_t j = 0; j < deg; ++j)
    if (!in_sorted(excl, nexcl, base + j)) elig[ne++] = j;
  int64_t n = 0;
  if (replace && fanout != -1) {
    const int64_t k = ne > 0 ? fanout : 0;
    for (int64_t t = 0; t < k; ++t) take[n++] = elig[mulhi64(x_key(seed, v, t), (uint64_t)ne)];
  } else {
    lpair_t* pairs = (lpair_t*)malloc(sizeof(lpair_t) * (size_t)(deg > 0 ? deg : 1));
    int64_t npos = 0;
    for (int64_t q = 0; q < ne; ++q) {
      const int64_t j = elig[q];
      if (pbytes) {
        const double w = widen(prob, pbytes, j);
        if (!sk_eligible(w)) continue;
        pairs[npos].key = oracle_weighted_key(seed, v, j, w);
      } else {
        pairs[npos].key = x_key(seed, v, j);
      }
      pairs[npos++].j = j;
    }
    const int64_t k = fanout == -1 ? npos : (npos < fanout ? npos : fanout);
    qsort(pairs, (size_t)npos, sizeof(lpair_t), cmp_lpair);
    char* chosen = (char*)calloc((size_t)(deg > 0 ? deg : 1), 1);
    for (int64_t t = 0; t < k; ++t) chosen[pairs[t].j] = 1;
    for (int64_t j = 0; j < deg; ++j)
      if (chosen[j]) take[n++] = j;
    free(chosen);
    free(pairs);
  }
  free(elig);
  return n;
}

/* Position of the first entry of row u equal to c (seg: the row's columns, `base` its first
 * position in A), or -1. */
static int64_t find_in_row(const int64_t* seg, int64_t deg, int64_t base, int64_t c) {
  for (int64_t j = 0; j < deg; ++j)
    if (seg[j] == c) return base + j;
  return -1;
}

/* ofspmm_edge_ids given the rows of the queries: query i looks in seg_col[seg_off[i], seg_off[i+1])
 * (empty for an out-of-range u), whose first position in A is seg_base[i]. */
void oracle_edge_ids(int64_t rows, const int64_t* u, const int64_t* v, int64_t n, const int64_t* seg_off,
                     const int64_t* seg_base, const int64_t* seg_col, int64_t* eid) {
  for (int64_t i = 0; i < n; ++i) {
    if (u[i] < 0 || u[i] >= rows) { eid[i] = -1; continue; }
    eid[i] = find_in_row(seg_col + seg_off[i], seg_off[i + 1] - seg_off[i], seg_base[i], v[i]);
  }
}

/* ofspmm_negative_sample given the rows of the sources: source i's row is seg_col[begin[i],
 * end[i]) (empty for an out-of-range source).  flags: 1 = reject edges of A, 2 = reject c == u. */
void oracle_negative_sample(int64_t rows, int64_t cols, const int64_t* src, int64_t num_src, const int64_t* begin,
                            const int64_t* end, const int64_t* seg_col, int64_t k, uint64_t seed, uint32_t flags,
                            int32_t max_trials, int64_t* neg, int64_t* counts) {
  counts[0] = counts[1] = 0;
  for (int64_t i = 0; i < num_src; ++i) {
    const int64_t u = src[i];
    const int valid = u >= 0 && u < rows;
    if (!valid) ++counts[1];
    for (int64_t t = 0; t < k; ++t) {
      int64_t c = -1;
      for (int32_t r = 0; valid && cols > 0 && r < max_trials; ++r) {
        const int64_t p = (int64_t)mulhi64(sk_mix64(sk_mix64(seed ^ (uint64_t)i) + (uint64_t)r * (uint64_t)k + (uint64_t)t),
                                           (uint64_t)cols);
        if ((flags & 2) && p == u) continue;
        if ((flags & 1) && find_in_row(seg_col + begin[i], end[i] - begin[i], 0, p) >= 0) continue;
        c = p;
        break;
      }
      if (c < 0) ++counts[0];
      neg[i * k + t] = c;
    }
  }
}
