// Shared helpers for the gll_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/gll_b200.h"

namespace gll {

void set_error(const char* fmt, ...);

#define GLL_CUDA_CHECK(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      gll::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return GLL_ERR_CUDA;                                                                \
    }                                                                                     \
  } while (0)

#define GLL_LAUNCH_CHECK()                                                                \
  do {                                                                                    \
    cudaError_t _e = cudaGetLastError();                                                  \
    if (_e != cudaSuccess) {                                                              \
      gll::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return GLL_ERR_CUDA;                                                                \
    }                                                                                     \
  } while (0)

#define GLL_REQUIRE(cond, msg)                \
  do {                                        \
    if (!(cond)) {                            \
      gll::set_error("%s (%s)", msg, #cond);  \
      return GLL_ERR_ARG;                     \
    }                                         \
  } while (0)

constexpr int WARP = 32;
constexpr unsigned FULL = 0xffffffffu;

__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// bump allocator over a caller-provided workspace
struct Carver {
  char* base;
  size_t off, cap;
  Carver(void* p, size_t bytes) : base((char*)p), off(0), cap(bytes) {}
  template <typename T>
  T* take(size_t count) {
    size_t o = align_up(off, 256);
    off = o + count * sizeof(T);
    return (T*)(base + o);
  }
  bool ok() const { return off <= cap; }
};

struct DeviceInfo {
  int device;
  int sms;
  int max_smem_optin;
};
const DeviceInfo& device_info();
// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute of a kernel: opt in once per (kernel, device),
// thread-safe (a process may drive several GPUs, e.g. the reference's nn.DataParallel, utils.py:547-548).
cudaError_t set_max_dynamic_smem_once(const void* func, int bytes);

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

// order-preserving map float -> uint32 (handles negatives), and back
__device__ __forceinline__ uint32_t float_to_ordered(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordered_to_float(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// ---- per-kernel launch counter and optional CUDA-event timing (gll_profile_* in the C ABI) ----
enum KernelId {
  KID_SQNORM = 0, KID_GRAM_TOPK, KID_GRAM_TOPK_TC, KID_RERANK, KID_KNN_FALLBACK, KID_GRAPH, KID_WEIGHTS, KID_CG, KID_PACK,
  KID_EDGE_GRAD, KID_ROW_GATHER, KID_CONVERT, KID_CG_ROWS, KID_LAPLACE_REFINE, KID_LAPLACE_FINISH,
  KID_KNN_SEGMENTS,   // segmented search: upload of seg_ptr and the unit table, per-row column windows
  KID_BATCH_REORDER,  // batched layer: kNN lists to the labeled-first order of the block-diagonal graph
  KID_LAPLACE_TRIALS_SETUP,  // laplace_learning_trials: the slot table of the labeled rows, index checks
  KID_COUNT
};
// RAII: counts the launch; when profiling is on, brackets it with two events on the launch stream.
struct ProfScope {
  int id;
  cudaStream_t st;
  void* slot;
  ProfScope(int id, cudaStream_t st);
  ~ProfScope();
};
#define GLL_PROF(id, st) gll::ProfScope _prof_scope_##id(gll::id, st)

// ---- internal launchers (one per stage), implemented in the .cu files ----
int knn_run(const float* X, int n, int d, int k, int row_begin, int row_end, int* knn_idx, float* knn_dist, int* info,
            void* ws, size_t ws_bytes, cudaStream_t st);
size_t knn_ws_bytes(int n, int d, int k, int row_begin, int row_end);
// base-set reuse across evaluation batches (knn.cu)
size_t knn_base_cache_bytes(int n_base);
int knn_base_cache_build(const float* Xbase, int n_base, int d, void* cache, void* ws, size_t ws_bytes, cudaStream_t st);
size_t knn_cached_ws_bytes(int n, int d, int k, int n_base);
int knn_run_cached(const float* X, int n, int d, int k, int n_base, const void* cache, int* knn_idx, float* knn_dist, int* info,
                   void* ws, size_t ws_bytes, cudaStream_t st);
// segmented search: independent graphs as row segments, seg_ptr on the host (knn.cu)
int knn_seg_check(int n, int d, int k, const int* seg_ptr, int nseg);
size_t knn_seg_ws_bytes(int n, int d, int k, const int* seg_ptr, int nseg);
int knn_run_segments(const float* X, int n, int d, int k, const int* seg_ptr, int nseg, int* knn_idx, float* knn_dist, int* info,
                     void* ws, size_t ws_bytes, cudaStream_t st);
void knn_seg_units(int n, int d, const int* seg_ptr, int nseg, long long* seg_units, long long* uniform_units);
void knn_tc_set_trace(void* device_buf);  // debug timeline of the Gram kernel's CTA 0 (knn_tc.cu)
int knn_debug_gram_tile(const float* X, int n, int d, int row_tile, int col_tile, float* acc_out, float* rscale_out, void* ws,
                        size_t ws_bytes, cudaStream_t st);

// One typed pointer per array of gll_layout: the graph, its system and the backward scratch, as the stages pass them on.
// The stage entry points fill only what they use and leave the rest NULL.
struct GraphBufs {
  int* knn_idx;
  float* knn_dist;
  int* row_ptr;
  int* col;
  float* dist;
  float* w;
  float* gv;
  float* eps;
  int* kappa;
  float* deg;
  float* bvec;
  int* uu_ptr;
  int* uu_col;
  float* uu_val;
  float* diag;
  float* rhs;
  float* ut;
  float* wt;
  int* info;
};
// the arrays of a state buffer laid out by gll_state_layout
GraphBufs graph_bufs(const gll_layout& L, void* state);

// K2 (phases 0-3: CSR with sorted rows) and K3 (phases 3-5: weights and the unlabeled system) as one cooperative launch over
// the phases [phase_begin, phase_end): 0-4 is K2, 3-6 K3 on sorted rows, 0-6 both (graph.cu)
int graph_stages_run(const GraphBufs& B, const float* Y, int n, int k, int l, int k_lab, int eps_auto, float eps_fixed, float tau,
                     int phase_begin, int phase_end, void* ws, size_t ws_bytes, cudaStream_t st);
size_t graph_ws_bytes(int n, int k);
// B stacked graphs of n rows (api.cu): the stage workspace of the batched drivers (the segmented search and its lists in natural
// order, the graph stages and the CG on the union; 0 for sizes the search refuses), and the segmented search itself followed by
// the reorder of its lists into B.knn_idx / B.knn_dist in labeled-first order
size_t batched_ws_bytes(int B, int n, int d, int k, int l, int k_lab);
int batched_knn_run(const float* X, int B, int n, int d, int k, int k_lab, const GraphBufs& G, void* ws, size_t ws_bytes, cudaStream_t st);
size_t weights_ws_bytes(int n, int k);
size_t graph_weights_ws_bytes(int n, int k);

// One CG solve (cg.cu).  Callers value-initialise it ({}) and set what they use by name.
struct CgSolve {
  // the system A = diag - offdiag(val) on m rows (compact CSR), rhs and x [m][lp] with lp = padded_classes(l)
  const int* ptr;
  const int* col;
  const float* val;
  const float* diag;
  const float* rhs;
  float* x;
  unsigned* ext_counter;  // optional [2], zero on entry: the on-chip kernel's grid barrier and exit ticket.  The kernel leaves
                          // both zero again, so one memset per forward (the info block) serves the forward AND the adjoint solve
  int* iters_out;         // device pointers, each may be NULL
  float* resid_out;
  int* status_out;
  // Fused conversions of the layer (the on-chip kernels do them in place; cg_run runs separate kernels for the others):
  const void* rhs_src;    // if set: the right-hand side is this [m][l] array (rhs_kind 1: fp32, 2: fp64); `rhs` is then scratch
  void* x_copy;           // if set: the solution is also written as an [m][l] array (fp64 if x_copy_f64, else fp32)
  const void* rhs_scale;  // optional device scalar (fp64 if rhs_scale_f64, else fp32) multiplied into rhs_src: the upstream gradient
                          // of a loss head whose d loss / d pred is rhs_src (losses.py: LaplaceLearningCELoss)
  int m, l, max_iter;
  float tol;  // > 0: absolute; < 0: |tol| times the largest column 2-norm of rhs
  int rhs_kind, x_copy_f64, rhs_scale_f64;
  float uu_degree_hint;  // expected off-diagonal entries per row of the system (0: unknown) -- picks the minibatch kernel
  // optional row mask of T trials x mask_cols columns (mask_col0: this solve's first column among them): A p is zeroed at (row i,
  // trial t) where mask_slot[i T + t] >= 0.  A masked solve always runs the streaming kernel.
  const int* mask_slot;
  int mask_trials, mask_cols, mask_col0;
};
int cg_run(const CgSolve& S, void* ws, size_t ws_bytes, cudaStream_t st);
// the unlabeled system of B with right-hand side B.rhs and the barrier words of B.info (which are zeroed with the info block)
inline CgSolve cg_system(const GraphBufs& B, int m, int l, float tol, int max_iter) {
  CgSolve S{};
  S.ptr = B.uu_ptr;
  S.col = B.uu_col;
  S.val = B.uu_val;
  S.diag = B.diag;
  S.m = m;
  S.rhs = B.rhs;
  S.l = l;
  S.tol = tol;
  S.max_iter = max_iter;
  S.ext_counter = (unsigned*)(B.info + GLL_INFO_CG_BARRIER);
  return S;
}
size_t cg_ws_bytes(int m, int l);
// the kernel cg_run takes for a system of m rows and lp <= CG_MAX_LP padded class columns: GLL_CG_KERNEL_*
int cg_pick(int m, int lp, float uu_degree_hint, bool masked);

// row-partitioned CG (cg_rows.cu): stage launchers.  peers == NULL: the host runs the NCCL collectives between them;
// otherwise the exchanges are fused into the kernels over peer memory (epoch = flag value of this stage, see cg_rows.cu)
size_t cg_rows_ws_bytes(int rows_local, int l);
size_t cg_rows_peer_mail_bytes();
size_t cg_rows_peer_flag_bytes();
int cg_rows_init(const float* diag, const float* rhs, int m, int l, int row_lo, int row_hi, float* x, float* u_full, void* ws,
                 size_t ws_bytes, const gll_peers* peers, unsigned epoch, cudaStream_t st);
int cg_rows_spmv(const int* uu_ptr, const int* uu_col, const float* uu_val, const float* diag, int m, int l, int row_lo, int row_hi,
                 const float* u_full, double* sums, void* ws, size_t ws_bytes, const gll_peers* peers, unsigned epoch,
                 const int* ctrl, cudaStream_t st);
int cg_rows_update(const float* diag, int m, int l, int row_lo, int row_hi, const double* sums, int iter, int max_iter, float tol,
                   float* x, float* u_full, int* ctrl, float* resid_out, void* ws, size_t ws_bytes, const gll_peers* peers,
                   unsigned epoch, cudaStream_t st);

// reads row_ptr, col, dist, w, eps, kappa, ut, wt of B; writes gv, bvec
int backward_edges_run(const float* X, int n, int d, int l, int k_lab, int eps_auto, const GraphBufs& B, float* dX, int row_begin,
                       int row_end, int phases, cudaStream_t st);

// column slices of m x lp class matrices (sharded solves): dst[r][c] = src[r][c0 + c] for c < cnt (zero padding), and back
int pack_columns(const float* src, int rows, int lp_src, int c0, int cnt, float* dst, int lp_dst, cudaStream_t st);
int unpack_columns(const float* src, int rows, int lp_src, int c0, int cnt, float* dst, int lp_dst, cudaStream_t st);


// small utility kernels (api.cu)
int pack_grad(const void* g, int is_f64, int m, int l, int lp, float* rhs, cudaStream_t st, float* zero_ptr = nullptr,
              long long zero_count = 0, const void* scale = nullptr, int scale_f64 = 0);
int unpack_pred(const float* ut_u, int m, int l, int lp, void* pred, int is_f64, cudaStream_t st);

inline int padded_classes(int l) { return (l + 3) / 4 * 4; }

}  // namespace gll
