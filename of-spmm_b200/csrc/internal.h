// internal.h — launcher interface between the C ABI (api.cu) and the per-op translation units.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <atomic>
#include <initializer_list>

#include "../../include/ofspmm.h"

namespace ofspmm {

#ifndef OFSPMM_ITEMS
#define OFSPMM_ITEMS 256
#endif
#ifndef OFSPMM_WARPS
#define OFSPMM_WARPS 4
#endif
constexpr int kTaskItems = OFSPMM_ITEMS;  // merge items (row-ends + non-zeros) per warp task
constexpr int kWarpsPerCta = OFSPMM_WARPS;

extern std::atomic<uint64_t> g_launches;
inline void count_launch(uint64_t k = 1) { g_launches.fetch_add(k, std::memory_order_relaxed); }

constexpr int kSmallTaskItems = 64;       // task size of the small-problem family
// Below this many 256-item tasks the machine (148 SMs x 36 resident warps) is not filled by one
// task per warp: AUTO switches to 64-item tasks so 4x more warps work in parallel.
constexpr int64_t kSmallProblemTasks = 148 * 36;

inline int64_t num_tasks(int64_t rows, int64_t nnz, int items = kTaskItems) {
  const int64_t total = rows + nnz;
  return (total + items - 1) / items;
}

// Matrices with at least this many non-zeros ("wide"; int64 indices only, int32 row offsets cannot
// hold them) keep 64-bit non-zero offsets in their task partition: 16-byte longlong2 entries
// instead of int2 (spmm_kernels.cuh:PartOf).  Below it every kernel runs exactly as with int2.
constexpr int64_t kWideNnz = (int64_t{1} << 31) - 1;
inline bool wide_nnz(int64_t nnz) { return nnz >= kWideNnz; }
inline size_t part_entry_bytes(int64_t nnz) { return wide_nnz(nnz) ? 16 : 8; }
// Task indices (task count x column panels) are drawn from a 32-bit counter and held in int; 2^30
// leaves room for the draws warps make past the last task.
constexpr int64_t kMaxTasks = int64_t{1} << 30;

// Resolved kernel family of a forward launch (public encoding: OFSPMM_VARIANT_*).
struct FwdVariant {
  int items;          // merge items per warp task: kTaskItems or kSmallTaskItems
  bool row_parallel;  // sub-warp per row (short rows, narrow dense operand) instead of nnz-parallel
  bool whole_rows;    // spmm_rows_kernel: one launch, no merge path (items = kSmallTaskItems for sizing)
};

// Elements in one 16-byte vector of a dense row (fp32: 4, bf16: 8).
constexpr int vec_width(size_t elem_bytes) { return static_cast<int>(16 / elem_bytes); }
inline int dense_vec_width(int dense_dtype) { return vec_width(dense_dtype == OFSPMM_DTYPE_BFLOAT16 ? 2 : 4); }

// The kernels whose lane layout follows the dense width n: the merge-path forward (256- and 64-item
// families; row-parallel family), the whole-row forward, the SDDMM (no layout: sddmm_wide_kernel)
// and the atomic A^T.dY scatter.
enum class LaneOp { kFwd, kFwdRowPar, kFwdRows, kSddmm, kAtomic };

// Template parameters of a kernel's lanes: LPR lanes span a dense row, each holding CH chunks of VEC
// elements; rows wider than one register tile (LPR * CH * VEC) run in `panels` column panels.
// lpr 0: the kernel has no layout for this width.  full: n is a whole number of register tiles.
struct LaneLayout {
  int vec = 1, lpr = 0, ch = 0, panels = 1;
  bool full = false;
  bool ok() const { return lpr != 0; }
};

// Lane layout of `op` for n dense columns.  `vec_ok`: the operands' addresses and strides allow
// 16-byte vector rows (n must also be a whole number of vectors).  Each op has its own ladders, one
// for vector and one for scalar lanes; a rung serves rows of up to `top` vectors (scalar lanes:
// elements), top 0 any wider row in column panels.
inline LaneLayout lane_layout(LaneOp op, int dense_dtype, int64_t n, bool vec_ok) {
  struct Rung { int64_t top; int lpr, ch; };
  const int w = dense_vec_width(dense_dtype);
  const bool vec = vec_ok && n % w == 0;
  const int64_t units = vec ? n / w : n;
  const int lane_vec = vec ? w : 1;
  auto pick = [&](std::initializer_list<Rung> ladder) {
    for (const Rung& r : ladder) {
      if (r.top != 0 && units > r.top) continue;
      const int64_t tile = int64_t{r.lpr} * r.ch;
      const int panels = r.top == 0 ? static_cast<int>((units + tile - 1) / tile) : 1;
      return LaneLayout{lane_vec, r.lpr, r.ch, panels, n % (tile * lane_vec) == 0};
    }
    return LaneLayout{lane_vec};
  };
  switch (op) {
    case LaneOp::kFwd:
      return vec ? pick({{8, 8, 1}, {16, 16, 1}, {32, 32, 1}, {64, 32, 2}, {0, 32, 4}})
                 : pick({{32, 32, 1}, {64, 32, 2}, {128, 32, 4}, {0, 32, 8}});
    case LaneOp::kFwdRowPar:  // sub-warp groups only
      return vec ? pick({{8, 8, 1}, {16, 16, 1}}) : pick({});
    case LaneOp::kFwdRows:
      return vec && n > 0 ? pick({{8, 8, 1}, {16, 16, 1}, {32, 32, 1}}) : pick({});
    case LaneOp::kSddmm:
      return vec ? pick({{8, 8, 1}, {16, 16, 1}, {32, 32, 1}, {64, 32, 2}, {128, 32, 4}})
                 : pick({{32, 32, 1}, {128, 32, 4}});
    case LaneOp::kAtomic:
      return vec ? pick({{8, 8, 1}, {16, 16, 1}, {32, 32, 1}, {64, 32, 2}, {0, 32, 4}})
                 : pick({{32, 32, 1}, {128, 32, 4}, {0, 32, 8}});
  }
  return pick({});
}

FwdVariant resolve_variant(int variant, int64_t rows, int64_t nnz, int64_t n, int dense_dtype);
struct FwdLaunch;
bool rows_kernel_applies(const ofspmm_csr* A, const void* B, int64_t ldb, const void* C, int64_t ldc, int64_t n,
                         int dense_dtype, const FwdLaunch& L);
int encode_variant(const FwdVariant& v);

// Per-launch options the C ABI passes down (ofspmm_opts).
struct FwdLaunch {
  FwdVariant variant;
  int tasks_per_warp;  // 0 = persistent grid
  int reserve_ctas;    // CTA slots per SM a persistent grid leaves free for overlapping exchange kernels
  bool dynamic;        // tasks drawn from a global counter (persistent grid only)
  bool wide;           // 64-bit non-zero offsets in the task partition (wide_nnz)
  unsigned flags;      // kFwd* epilogue bits
  const void* bias;
  float* acc32;        // fp32 accumulator of multi-pass 16-bit products
};
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct DevInfo {
  int sms;
  int cc_major;
  int ordinal;
};

// Launch constants of one kernel instantiation per device ordinal (0 = not queried yet); values
// are immutable once written, relaxed atomics make concurrent first calls benign.
struct KernelLaunchCache {
  static constexpr int kMaxDevices = 64;
  std::atomic<int> occ[kMaxDevices];
  KernelLaunchCache() { for (auto& o : occ) o.store(0, std::memory_order_relaxed); }
  int get(int dev) const { return dev >= 0 && dev < kMaxDevices ? occ[dev].load(std::memory_order_relaxed) : 0; }
  void set(int dev, int v) { if (dev >= 0 && dev < kMaxDevices) occ[dev].store(v, std::memory_order_relaxed); }
};
int get_dev_info(DevInfo* out);  // OFSPMM_OK / OFSPMM_ERR_CUDA

// Layout of the workspace shared by fwd / bwd(transpose) calls.
struct FwdWorkspace {
  size_t counter_off, part_off, carry_off, head_off, total;
};
FwdWorkspace fwd_workspace_layout(int64_t rows, int64_t nnz, int64_t n, int dense_dtype, int items = kTaskItems);

// Each returns an OFSPMM_* status; all launches go to `stream`.
int launch_task_partition(const void* crow, int idx_dtype, int64_t rows, int64_t nnz, int64_t P,
                          int items, void* part, cudaStream_t stream);
int launch_fwd(const ofspmm_csr* A, const void* B, int64_t ldb, void* C, int64_t ldc, int64_t n,
               int dense_dtype, const void* part, float* carry, float* head, void* counter, int64_t P,
               const FwdLaunch& L, cudaStream_t stream);
int launch_sddmm(const ofspmm_csr* A, const void* dY, const void* B, void* dval, int64_t n,
                 int dense_dtype, const void* part, void* counter, int64_t P, cudaStream_t stream);
int launch_bwd_atomic(const ofspmm_csr* A, const void* dY, float* acc, void* dB_cast_out,
                      int64_t n, int dense_dtype, const void* part, int64_t P, cudaStream_t stream);
int launch_partition_public(const void* crow, int idx_dtype, int64_t rows, int64_t nnz,
                            int64_t parts, int64_t* out_row, int64_t* out_nz, cudaStream_t stream);
int launch_row_hist(const void* crow, int idx_dtype, int64_t rows, int64_t* hist32,
                    cudaStream_t stream);
size_t transpose_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int idx_dtype);
int launch_transpose(const ofspmm_csr* A, void* t_crow, void* t_col, void* t_val, void* t_perm,
                     void* ws, size_t ws_bytes, cudaStream_t stream);
const char* fwd_variant_name(int64_t n, int dense_dtype, bool aligned);
size_t coo_to_csr_workspace_bytes(int64_t n, int64_t rows, int64_t cols);
int launch_coo_to_csr(const int64_t* row, const int64_t* col, const float* val, int64_t n, int64_t rows, int64_t cols,
                      int mode, int idx_dtype, void* crow, void* col_out, float* val_out, int64_t* counts, void* ws,
                      size_t ws_bytes, cudaStream_t stream);
size_t sample_neighbors_workspace_bytes(int64_t num_dst, int64_t cap);
int launch_sample_neighbors(const ofspmm_csr* A, const void* dst, int64_t num_dst, int64_t fanout, uint64_t seed,
                            int64_t cap, void* blk_crow, void* blk_col, void* blk_val, void* src_nodes, int64_t* counts,
                            void* ws, cudaStream_t stream);
int launch_expand_rows(const void* crow, int idx_dtype, int64_t rows, int64_t* out, cudaStream_t stream);
int launch_csr_normalize(const void* crow, const void* col, float* val, int idx_dtype, int64_t rows, int64_t cols, int mode,
                         float* dinv, cudaStream_t stream);
int launch_gather_vals(const void* val, int val_dtype, const void* perm, int idx_dtype, int64_t nnz,
                       void* out, cudaStream_t stream);
int launch_gather_rows(void* dst, int64_t ld_dst, const void* src, int64_t ld_src, const void* list,
                       int idx_dtype, int64_t idx_offset, int64_t count, int64_t n, int dense_dtype,
                       int max_ctas, cudaStream_t stream);
int launch_scatter_add_rows_f32(float* dst, int64_t ld_dst, const void* src, int64_t ld_src, const void* list,
                                int idx_dtype, int64_t idx_offset, int64_t count, int64_t n, int src_dtype,
                                int max_ctas, cudaStream_t stream);
int launch_signal_peers(void* const* slots, int n, unsigned long long epoch, cudaStream_t stream);
int launch_pull_rows_multi(void* dst, int64_t ld_dst, int64_t ld_src, const ofspmm_pull_seg* segs, int nseg,
                           unsigned long long epoch, int64_t n, int dense_dtype, int idx_dtype, int max_ctas,
                           cudaStream_t stream);
int launch_combine_rows_multi(float* acc, int64_t ld_acc, int64_t ld_src, const ofspmm_combine_seg* segs, int nseg,
                              unsigned long long epoch, int64_t rows, int64_t n, int src_dtype, int max_ctas,
                              cudaStream_t stream);
int launch_cast_from_f32(const float* src, void* dst, int64_t count, int dst_dtype, cudaStream_t stream);
int launch_scatter_add_rows(void* dst, int64_t ld_dst, const void* src, int64_t ld_src, const void* list,
                            int idx_dtype, int64_t idx_offset, int64_t count, int64_t n, int dense_dtype,
                            int max_ctas, cudaStream_t stream);

#define OFSPMM_CUDA_OK(expr)                         \
  do {                                               \
    if ((expr) != cudaSuccess) return OFSPMM_ERR_CUDA; \
  } while (0)

}  // namespace ofspmm
