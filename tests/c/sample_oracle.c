/*
 * sample_oracle.c — CPU restatement of neighbour sampling (ofspmm_sample_neighbors,
 * include/ofspmm.h).  TEST INFRASTRUCTURE ONLY: tests/_sample_oracle.py compiles it with gcc into a
 * temporary directory and loads it; the product package never does.
 *
 * It follows the definition step by step rather than the device algorithm: every key of a row is
 * computed and sorted, the first k are taken, out-of-range columns are dropped, then the sampled ids
 * are relabelled.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>


/* The sampler's key mixer: multiply by 0x9E3779B97F4A7C15, then the splitmix64 finaliser. */
static uint64_t sample_mix64(uint64_t x) {
  x *= 0x9E3779B97F4A7C15ull;
  x ^= x >> 30;
  x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27;
  x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return x;
}

/* key(s, v, j) = mix(mix(s ^ v) + j), all mod 2^64. */
uint64_t oracle_sample_key(uint64_t seed, int64_t v, int64_t j) {
  return sample_mix64(sample_mix64(seed ^ (uint64_t)v) + (uint64_t)j);
}

typedef struct { uint64_t key; int64_t j; } sample_pair;

static int cmp_pair(const void* a, const void* b) {
  const sample_pair* x = (const sample_pair*)a;
  const sample_pair* y = (const sample_pair*)b;
  if (x->key != y->key) return x->key < y->key ? -1 : 1;
  return x->j < y->j ? -1 : (x->j > y->j);
}

static int cmp_i64(const void* a, const void* b) {
  const int64_t x = *(const int64_t*)a, y = *(const int64_t*)b;
  return x < y ? -1 : (x > y);
}

/* occurrences of x in the sorted array a[n] */
static int64_t count_sorted(const int64_t* a, int64_t n, int64_t x, int64_t* first) {
  int64_t lo = 0, hi = n;
  while (lo < hi) { const int64_t mid = (lo + hi) / 2; if (a[mid] < x) lo = mid + 1; else hi = mid; }
  *first = lo;
  int64_t e = lo;
  while (e < n && a[e] == x) ++e;
  return e - lo;
}

/* ofspmm_sample_neighbors (include/ofspmm.h) restated literally, for a square A of `rows` rows.
 * The rows are given per destination, so that a matrix too large for the host can be checked from
 * its destinations' rows alone: the entries of row dst[i] are seg_col / seg_val at
 * [seg_off[i], seg_off[i+1]) (ignored for an invalid destination).  vbytes: bytes per value (0 for a
 * pattern matrix, 2 for bf16, 4 for fp32), copied bit for bit.  The caller sizes blk_col / blk_val
 * for the sum of k and src_nodes for num_dst + that sum.  counts as in the header. */
void oracle_sample_neighbors(int64_t rows, const int64_t* dst, int64_t num_dst, const int64_t* seg_off,
                             const int64_t* seg_col, const void* seg_val, int vbytes, int64_t fanout, uint64_t seed,
                             int64_t* blk_crow, int64_t* blk_col, void* blk_val, int64_t* src_nodes, int64_t* counts) {
  int64_t* sdst = (int64_t*)malloc(sizeof(int64_t) * (size_t)(num_dst > 0 ? num_dst : 1));
  memcpy(sdst, dst, sizeof(int64_t) * (size_t)num_dst);
  qsort(sdst, (size_t)num_dst, sizeof(int64_t), cmp_i64);
  int64_t nnz = 0, invalid = 0, first = 0;
  blk_crow[0] = 0;
  for (int64_t i = 0; i < num_dst; ++i) {
    const int64_t v = dst[i];
    /* a destination is valid when it is a row of A and occurs once in dst */
    if (v < 0 || v >= rows || count_sorted(sdst, num_dst, v, &first) != 1) {
      ++invalid;
      blk_crow[i + 1] = nnz;
      continue;
    }
    const int64_t b = seg_off[i], deg = seg_off[i + 1] - b;
    const int64_t k = fanout == -1 ? deg : (deg < fanout ? deg : fanout);
    /* every key of the row, sorted by (key, j); the first k are selected */
    sample_pair* pairs = (sample_pair*)malloc(sizeof(sample_pair) * (size_t)(deg > 0 ? deg : 1));
    char* chosen = (char*)calloc((size_t)(deg > 0 ? deg : 1), 1);
    for (int64_t j = 0; j < deg; ++j) { pairs[j].key = oracle_sample_key(seed, v, j); pairs[j].j = j; }
    qsort(pairs, (size_t)deg, sizeof(sample_pair), cmp_pair);
    for (int64_t t = 0; t < k; ++t) chosen[pairs[t].j] = 1;
    /* in ascending j, without the entries whose column lies outside [0, cols) (cols == rows) */
    for (int64_t j = 0; j < deg; ++j) {
      const int64_t c = seg_col[b + j];
      if (!chosen[j] || c < 0 || c >= rows) continue;
      blk_col[nnz] = c;   /* global id for now, relabelled below */
      if (vbytes) memcpy((char*)blk_val + nnz * vbytes, (const char*)seg_val + (b + j) * vbytes, (size_t)vbytes);
      ++nnz;
    }
    blk_crow[i + 1] = nnz;
    free(pairs);
    free(chosen);
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
  sample_pair* where = (sample_pair*)malloc(sizeof(sample_pair) * (size_t)(num_dst > 0 ? num_dst : 1));
  for (int64_t i = 0; i < num_dst; ++i) { where[i].key = (uint64_t)dst[i]; where[i].j = i; }
  qsort(where, (size_t)num_dst, sizeof(sample_pair), cmp_pair);
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
