/* gll_b200.h -- C ABI of libgll_b200.so: the B200 (sm_100a) implementation of the GraphLearningLayer
 * hot path (forward + backward of LaplaceLearningSparseHard).
 *
 * The reference (pure Python, /root/reference/GLL.py) has no FFI; every entry point below cites the
 * reference code it replaces.  Conventions for ALL entry points:
 *   - plain pointers and sizes only; every array pointer is a DEVICE pointer unless it says "host";
 *   - dense matrices row-major, fp32 values, int32 indices;
 *   - the library never allocates or frees device memory: the caller passes a workspace
 *     (size from the matching *_workspace_bytes query) and owns every buffer;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work is
 *     enqueued on it and nothing synchronises with the host unless stated;
 *   - return value 0 = success, negative = error (gll_last_error() gives a thread-local message).
 *   - labeled ("base") nodes are the FIRST k_lab rows (GLL.py:11,32-38).
 */
#ifndef GLL_B200_H
#define GLL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GLL_OK 0
#define GLL_ERR_ARG (-1)      /* bad argument (null pointer, unsupported size) */
#define GLL_ERR_WORKSPACE (-2) /* workspace too small */
#define GLL_ERR_CUDA (-3)     /* a CUDA runtime call failed */

/* bits of info[GLL_INFO_STATUS] */
#define GLL_STATUS_CG_NOT_CONVERGED 1 /* GLL.py:273-274 prints 'max iter reached' */
#define GLL_STATUS_EPS_TINY 2         /* GLL.py:240-241 warns "Epsilon in KNN is very close to zero." */
#define GLL_STATUS_NONFINITE 4
#define GLL_STATUS_KNN_FALLBACK 8     /* some rows needed the exact brute-force kNN fallback (informational) */
#define GLL_STATUS_BAD_INDEX 16       /* gll_laplace_eval_trials: a trial's labeled-row index is outside [0, n) or repeated */

/* slots of the int32 info[16] block that lives in the state buffer */
#define GLL_INFO_STATUS 0
#define GLL_INFO_NNZ 1        /* E: directed edges of the symmetrised graph */
#define GLL_INFO_NNZ_UU 2     /* off-diagonal nnz of L_uu */
#define GLL_INFO_CG_ITERS_FWD 3
#define GLL_INFO_CG_ITERS_BWD 4
#define GLL_INFO_KNN_FALLBACK_ROWS 5
#define GLL_INFO_CG_RESID_FWD 6 /* float bits: max_c ||r_c||_2 at exit */
#define GLL_INFO_CG_RESID_BWD 7
/* gll_laplace_eval only */
#define GLL_INFO_LAPLACE_ROUNDS 8       /* refinement rounds that ran a correction solve */
#define GLL_INFO_LAPLACE_CG_ITERS 9     /* correction-CG iterations, all rounds */
#define GLL_INFO_LAPLACE_RESID 10       /* float bits: max_c ||M r_c||_2 at the last refinement round */
#define GLL_INFO_LAPLACE_RESID0 11      /* float bits: the same after the initial solve */
#define GLL_INFO_CG_BARRIER 12          /* two words, every fused call: the on-chip CG's grid barrier (zeroed with info, rewound by the kernel) */
#define GLL_INFO_LAPLACE_ROUND_ITERS 14 /* two words: correction-CG iterations of round r in bits [16 (r % 2), +16) of word 14 + r / 2 */
#define GLL_INFO_WORDS 16

/* gll_laplace_eval's refinement schedule (chosen from the CPU model in tests/test_laplace_eval_cpu.py): the initial fp32 solve
 * stops at GLL_LAPLACE_CG_RTOL0 times its right-hand side's largest column norm, each correction solve at GLL_LAPLACE_CG_RTOL,
 * and GLL_LAPLACE_ROUNDS fp64 residual rounds run. */
#define GLL_LAPLACE_ROUNDS 4
#define GLL_LAPLACE_CG_RTOL0 1e-5
#define GLL_LAPLACE_CG_RTOL 1e-4

const char* gll_last_error(void);
int gll_version(void);
/* number of SMs / device ordinal the library sees for the current device (host query). */
int gll_device_sm_count(void);

/* Launch accounting and optional per-kernel timing (used by bench.py; off by default).  Every kernel launch of
 * the library increments a counter; gll_launch_count(id) reads one kernel's counter, id < 0 the total.  With
 * gll_profile_enable(1) each launch is bracketed by two CUDA events on its own stream; gll_profile_collect()
 * synchronises on them, writes per-kernel summed milliseconds and launch counts (arrays of gll_kernel_count()
 * entries, either may be NULL) and clears the records. */
int gll_kernel_count(void);
const char* gll_kernel_name(int id);
long long gll_launch_count(int id);
void gll_profile_enable(int on);
int gll_profile_collect(double* ms_sum, long long* count);
/* Debug aid: when device_buf != NULL the on-chip CG kernel writes %globaltimer stamps [cta][16 passes][8 phases]
 * (uint64) into it; NULL switches the trace off.  Not for production use. */
void gll_debug_cg_trace(void* device_buf);
/* Debug aid: SM-clock timeline of CTA 0 of the tensor-core Gram kernel, [4 warps][1024 units][8 phases] uint64
 * (MMA warp, two epilogue warps, TMA producer; tools/knn_trace.py); NULL switches it off.  Not for production use. */
void gll_debug_knn_trace(void* device_buf);

/* Class columns are padded to a multiple of 4 so that every class row is float4-addressable. */
int gll_padded_classes(int l);
/* Upper bound of directed edges: 2*n*(k-1). */
size_t gll_max_edges(int n, int k);

/* ---------------------------------------------------------------------------------------------
 * Byte offsets (256-B aligned) of the arrays kept between forward and backward.  Replaces the Python
 * attributes the reference stores on ctx (GLL.py:69-70: W, V, Luu, label_matrix, mod_V, C, knn_ind, X, Pred).
 * ------------------------------------------------------------------------------------------- */
typedef struct gll_layout {
  size_t knn_idx;  /* int32 [n*k]      kNN lists, self in slot 0              (GLL.py:183) */
  size_t knn_dist; /* float [n*k]      distances, fp32                        (GLL.py:183) */
  size_t row_ptr;  /* int32 [n+1]      CSR of the symmetrised graph           (GLL.py:196-198) */
  size_t col;      /* int32 [Emax]     sorted within each row */
  size_t dist;     /* float [Emax]     one distance per undirected edge */
  size_t w;        /* float [Emax]     W_ij = exp(-4 d^2/(eps_i eps_j))        (GLL.py:216,233) */
  size_t gv;       /* float [Emax]     backward scratch: G_ij * V_ij           (GLL.py:146) */
  size_t eps;      /* float [n]        bandwidths                             (GLL.py:205,226) */
  size_t kappa;    /* int32 [n]        kappa(i) = last kNN entry (replaces the dense C, GLL.py:209-213) */
  size_t deg;      /* float [n]        degree = row sum of W                   (GLL.py:29) */
  size_t bvec;     /* float [n]        backward: b_i = sum_j G_ij modV_ij      (GLL.py:126) */
  size_t uu_ptr;   /* int32 [m+1]      compact CSR of the off-diagonal of L_uu (GLL.py:37) */
  size_t uu_col;   /* int32 [Emax]     column index rebased to the unlabeled block */
  size_t uu_val;   /* float [Emax]     W_ij (the solver applies diag*p - sum W p) */
  size_t diag;     /* float [m]        deg_i + tau                             (GLL.py:48) */
  size_t rhs;      /* float [m*lp]     B = -L_ul Y, later the adjoint rhs      (GLL.py:53,93) */
  size_t ut;       /* float [n*lp]     [Y; Pred]                               (GLL.py:109) */
  size_t wt;       /* float [n*lp]     [0; w]                                  (GLL.py:104) */
  size_t info;     /* int32 [GLL_INFO_WORDS] */
  size_t total;    /* bytes to allocate */
} gll_layout;

int gll_state_layout(int n, int k, int l, int k_lab, gll_layout* out);
size_t gll_workspace_bytes(int n, int d, int k, int l, int k_lab);

/* ---------------------------------------------------------------------------------------------
 * Stage entry points (each is also what the parity tests call)
 * ------------------------------------------------------------------------------------------- */

/* K1. Exact k nearest neighbours (2 <= k <= 64; k > 33 runs two candidate rounds and needs n >= 256) of every row of X (n x d), Euclidean, self in slot 0 with distance 0,
 * remaining slots ordered by (distance, index).  Replaces gl.weightmatrix.knnsearch(...,'annoy') at
 * GLL.py:181-189.  Candidate selection runs as a tiled Gram GEMM with a fused per-row top-k epilogue (the
 * n x n matrix never reaches HBM); kept distances are recomputed as sqrt(sum (x_i-x_j)^2) in fp64 and
 * rounded to fp32; rows whose candidate set cannot be proven complete are redone by brute force.
 * info may be NULL; otherwise info[GLL_INFO_KNN_FALLBACK_ROWS] / GLL_STATUS_KNN_FALLBACK are updated. */
size_t gll_knn_workspace_bytes(int n, int d, int k);
int gll_knn(const float* X, int n, int d, int k, int* knn_idx, float* knn_dist, int* info,
            void* workspace, size_t workspace_bytes, void* stream);

/* K1 over independent graphs stacked as row segments: segment s is rows [seg_ptr_host[s], seg_ptr_host[s+1]) of X (n x d),
 * seg_ptr_host a HOST array of nseg + 1 offsets from 0 to n (the search is planned on the host: no sync).  Row i of segment s
 * gets its k nearest neighbours among the rows of s only (global row numbers, self in slot 0, then by (distance, index)):
 * bit-identical to gll_knn on each segment alone plus the segment's offset, because those lists are exact.  Every segment
 * needs >= k rows; 2 <= k <= 64, with n >= 256 when k > 33 (as gll_knn: k > 33 runs two tensor-core candidate rounds,
 * the second above the first round's 32nd key).  The tensor-core search only issues the (row tile, column tile) units whose
 * columns meet the segments of the tile's rows, O(sum n_s^2 d) work instead of O(n^2 d).  nseg == 1 runs gll_knn.  Bad arguments
 * return GLL_ERR_ARG before any CUDA call; the workspace query returns 0 for them.  gll_knn_segments_units (host query,
 * for benchmarks): tensor-core units such a call issues, and those of the uniform grid over the same rows (0, 0 when
 * the SIMT path runs). */
size_t gll_knn_segments_workspace_bytes(int n, int d, int k, const int* seg_ptr_host, int nseg);
int gll_knn_segments(const float* X, int n, int d, int k, const int* seg_ptr_host, int nseg, int* knn_idx, float* knn_dist,
                     int* info, void* workspace, size_t workspace_bytes, void* stream);
void gll_knn_segments_units(int n, int d, const int* seg_ptr_host, int nseg, long long* seg_units, long long* uniform_units);

/* K2. Symmetrise (elementwise max == union graph) and build the CSR; zero distances and self loops are
 * not edges.  Replaces the scipy sequence at GLL.py:192-198. col/dist need gll_max_edges(n,k) entries. */
size_t gll_graph_workspace_bytes(int n, int k);
int gll_graph_build(const int* knn_idx, const float* knn_dist, int n, int k, int* row_ptr, int* col,
                    float* dist, int* info, void* workspace, size_t workspace_bytes, void* stream);

/* K3. Bandwidths, weights, degree, and the linear system of the unlabeled block.
 * eps_auto != 0: eps_i = knn_dist[i][k-1], kappa_i = knn_idx[i][k-1] (GLL.py:205-211); else eps_i = eps_fixed
 * (GLL.py:226).  W (GLL.py:216/233), deg (GLL.py:29), diag = deg + tau, compact off-diagonal CSR of
 * L_uu (GLL.py:37,48), rhs = W_ul Y = -L_ul Y (GLL.py:53), and ut[:k_lab] = Y.  Y is k_lab x l fp32. */
size_t gll_weights_workspace_bytes(int n, int k);
int gll_edge_weights(const int* knn_idx, const float* knn_dist, const int* row_ptr, const int* col,
                     const float* dist, const float* Y, int n, int k, int l, int k_lab, int eps_auto,
                     float eps_fixed, float tau, float* eps, int* kappa, float* w, float* deg, int* uu_ptr,
                     int* uu_col, float* uu_val, float* diag, float* rhs, float* ut, int* info,
                     void* workspace, size_t workspace_bytes, void* stream);

/* K4. Multi-right-hand-side Jacobi-preconditioned CG on A = diag - offdiag(uu_val), x0 = 0, all class
 * columns at once, per-column freeze and absolute 2-norm stop like stable_conjgrad (GLL.py:247-276; the
 * p = r alias of GLL.py:254 is not reproduced).  Replaces spsolve at GLL.py:53 and GLL.py:93.
 * tol > 0: absolute (the reference's meaning); tol < 0: |tol| times the largest column 2-norm of rhs.
 * One persistent cooperative launch runs all iterations.  rhs and x are m x lp (lp = padded classes);
 * x may alias nothing else.  iters_out / resid_out are device pointers (may be NULL). */
size_t gll_cg_workspace_bytes(int m, int l);
int gll_cg_solve(const int* uu_ptr, const int* uu_col, const float* uu_val, const float* diag,
                 const float* rhs, int m, int l, float tol, int max_iter, float* x, int* iters_out,
                 float* resid_out, int* status_out, void* workspace, size_t workspace_bytes, void* stream);
/* The same with the caller's expectation of off-diagonal entries per row (0: unknown).  The solver cannot see nnz from the host;
 * sparse minibatch systems (up to 5 entries per row, 64..2048 rows) take the thread-block-cluster kernel.  gll_forward /
 * gll_backward pass 1.2 (k - 1) m / n; a caller that wants bit-identical results to the layer passes the same number. */
int gll_cg_solve_hint(const int* uu_ptr, const int* uu_col, const float* uu_val, const float* diag,
                      const float* rhs, int m, int l, float tol, int max_iter, float* x, int* iters_out,
                      float* resid_out, int* status_out, void* workspace, size_t workspace_bytes, void* stream,
                      float uu_degree_hint);
/* Host-only query (no GPU needed): the kernel gll_cg_solve_hint runs for m rows, 1 <= l <= 128 class columns and the hint,
 * under the current GLL_B200_CG_PATH; GLL_ERR_ARG outside that range.  More than 128 columns are solved in chunks of 128, each
 * picked on its own without the hint. */
#define GLL_CG_KERNEL_STREAMING 0 /* vectors in global memory, any size */
#define GLL_CG_KERNEL_RESIDENT 1  /* multi-CTA, vectors and matrix slices in shared memory */
#define GLL_CG_KERNEL_SMALL 2     /* one CTA, up to 512 rows */
#define GLL_CG_KERNEL_CLUSTER 3   /* one cluster of eight CTAs, 64 to 2048 rows, sparse systems */
int gll_cg_kernel(int m, int l, float uu_degree_hint);

/* K5+K6. Backward edge pass (GLL.py:104-159): G_ij = -<wt_i-wt_j, ut_i-ut_j>, gv = G*V, b_i = sum_j G_ij modV_ij
 * (auto only), dX_i = sum_j t_ij (x_i - x_j) with t_ij = gv_ij - [j==kappa(i)] b_i - [kappa(j)==i] b_j. */
int gll_backward_edges(const float* X, int n, int d, int l, int k_lab, int eps_auto, const int* row_ptr,
                       const int* col, const float* dist, const float* w, const float* eps, const int* kappa,
                       const float* ut, const float* wt, float* gv, float* bvec, float* dX, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Row-range and column-slice variants: the building blocks of the sharded (one graph on N GPUs) path, see
 * graphlearninglayer_b200/sharded.py.  Nodes are sharded by ROWS for the kNN search and the backward gather (results are
 * all-gathered by the host with NCCL); the two CG solves are sharded by CLASS COLUMNS (columns of the multi-RHS CG are
 * independent, GLL.py:262-269, so no communication happens inside the solver).
 * ------------------------------------------------------------------------------------------- */
/* gll_knn for rows [row_begin, row_end) against all n columns; writes rows [row_begin, row_end) of the full n x k
 * arrays.  row_begin should be a multiple of 128 (otherwise the SIMT Gram path is taken). */
/* Verification only: the raw fp32 accumulator acc_out[128][256] that the tensor-core kNN kernel forms for rows
 * [128 row_tile, +128) against columns [256 col_tile, +256) from the split operands (mode of GLL_B200_KNN_SPLIT), and the
 * operands' per-row scale rscale_out[n] (the accumulator holds x_i.x_j / (rscale_i rscale_j)).
 * tests compare it with the numpy model of the split (oracle/split_model.py).  workspace: gll_knn_workspace_bytes(n, d, 25). */
int gll_debug_gram_tile(const float* X, int n, int d, int row_tile, int col_tile, float* acc_out, float* rscale_out,
                        void* workspace, size_t workspace_bytes, void* stream);
/* Base-set reuse across evaluation batches (utils.py:596-621, test_network: the layer is called on [base; test batch]
 * with the SAME base rows for every batch; SURVEY.md 8f-4).  gll_base_cache_build searches the n_base base rows among
 * themselves once and keeps, per base row, its 32 best base columns (cache: gll_base_cache_bytes(n_base) bytes of device
 * memory owned by the caller).  gll_knn_cached is gll_knn(X, n, ...) for X = [base (n_base rows, the ones the cache was built
 * from); batch] that searches only the batch rows against all columns and the base rows against the batch columns; the
 * emitted lists are identical to gll_knn's (same exact re-rank and completeness proof).  n_base >= 256, k <= 33. */
size_t gll_base_cache_bytes(int n_base);
size_t gll_base_cache_workspace_bytes(int n_base, int d);
int gll_base_cache_build(const float* Xbase, int n_base, int d, void* cache, void* workspace, size_t workspace_bytes,
                         void* stream);
size_t gll_knn_cached_workspace_bytes(int n, int d, int k, int n_base);
int gll_knn_cached(const float* X, int n, int d, int k, int n_base, const void* cache, int* knn_idx, float* knn_dist,
                   int* info, void* workspace, size_t workspace_bytes, void* stream);
size_t gll_knn_rows_workspace_bytes(int n, int d, int k, int row_begin, int row_end);
int gll_knn_rows(const float* X, int n, int d, int k, int row_begin, int row_end, int* knn_idx, float* knn_dist, int* info,
                 void* workspace, size_t workspace_bytes, void* stream);
/* gll_backward_edges restricted to rows [row_begin, row_end); phases bit 0: K5 (gv of the rows' edges, b of the rows),
 * bit 1: K6 (dX rows; reads b of ALL rows, i.e. after the host has gathered bvec). */
int gll_backward_edges_rows(const float* X, int n, int d, int l, int k_lab, int eps_auto, const int* row_ptr, const int* col,
                            const float* dist, const float* w, const float* eps, const int* kappa, const float* ut,
                            const float* wt, float* gv, float* bvec, float* dX, int row_begin, int row_end, int phases,
                            void* stream);
/* dst[r][c] = src[r][c0 + c] for c < cnt, zero for cnt <= c < lp_dst (rows x lp_src -> rows x lp_dst), and the inverse
 * (dst[r][c0 + c] = src[r][c], c < cnt). */
int gll_pack_columns(const float* src, int rows, int lp_src, int c0, int cnt, float* dst, int lp_dst, void* stream);
int gll_unpack_columns(const float* src, int rows, int lp_src, int c0, int cnt, float* dst, int lp_dst, void* stream);
/* K4 for ONE graph whose unlabeled rows are partitioned over ranks (BASELINE north star: "row-block partitioned, CG
 * iterate exchanged by all-gather, dot products by all-reduce").  The library does not link NCCL: these are the three
 * per-rank stages and the host runs the two collectives between them on the same stream
 * (graphlearninglayer_b200/sharded.py: torch.distributed all_gather_into_tensor / all_reduce):
 *     init;  repeat { all-gather u_full;  spmv -> sums[3*lp] (fp64: <r,u>, <w,u>, <r,r> over own rows);
 *                     all-reduce(sum) sums;  update(iter) }  until ctrl[0] != 0.
 * Arithmetic: Jacobi-preconditioned Chronopoulos-Gear CG, per-column freeze / stop test of stable_conjgrad
 * (GLL.py:247-276), identical on every rank because every rank sees the same reduced sums.
 * x, u_full: m' x lp with m' >= m (rows [row_lo,row_hi) are written; u_full is the all-gather buffer).
 * ctrl: int[4] zeroed by the caller: [0] stop flag, [1] iterations, [2] GLL_STATUS_* bits.  The workspace keeps r, p, s, w
 * of the own rows between calls and must not be touched while a solve is running. */
size_t gll_cg_rows_workspace_bytes(int rows_local, int l);
int gll_cg_rows_init(const float* diag, const float* rhs, int m, int l, int row_lo, int row_hi, float* x, float* u_full,
                     void* workspace, size_t workspace_bytes, void* stream);
int gll_cg_rows_spmv(const int* uu_ptr, const int* uu_col, const float* uu_val, const float* diag, int m, int l, int row_lo,
                     int row_hi, const float* u_full, double* sums, void* workspace, size_t workspace_bytes, void* stream);
int gll_cg_rows_update(const float* diag, int m, int l, int row_lo, int row_hi, const double* sums, int iter, int max_iter,
                       float tol, float* x, float* u_full, int* ctrl, float* resid_out, void* workspace, size_t workspace_bytes,
                       void* stream);
/* Peer-memory mode of the same three stages: the all-gather and the all-reduce are fused INTO the kernels over NVLink peer
 * pointers (symmetric memory: every rank maps every rank's buffers), so the loop needs no NCCL call and no host round trip:
 * update/init store the new u rows into every rank's u array and raise an epoch flag on every peer; spmv waits on its
 * LOCAL flags for everybody's u, writes its partial sums into a mailbox row on every peer and raises a second flag; update
 * waits for all sums and adds the mailbox rows in rank order.  Flags only grow: the caller supplies `epoch` values that
 * increase monotonically over the life of the buffers (init: e; iteration it: spmv and update both e + it; the next solve
 * starts above e + iterations + 1).  peers->u[p] / mail[p] / flags[p]: rank p's u array (m' x lp fp32), mailbox
 * (gll_cg_rows_peer_mail_bytes()) and flag block (gll_cg_rows_peer_flag_bytes(), zeroed once before first use), as mapped
 * in THIS process; p = 0..world-1 <= 8, own rank included.  Every rank must enqueue the same sequence of launches; a wait
 * longer than 2 s traps the kernel instead of hanging the GPU. */
typedef struct gll_peers {
  void* u[8];
  void* mail[8];
  void* flags[8];
  int world;
  int rank;
} gll_peers;
size_t gll_cg_rows_peer_mail_bytes(void);
size_t gll_cg_rows_peer_flag_bytes(void);
int gll_cg_rows_init_p2p(const float* diag, const float* rhs, int m, int l, int row_lo, int row_hi, float* x,
                         const gll_peers* peers, unsigned epoch, void* workspace, size_t workspace_bytes, void* stream);
int gll_cg_rows_spmv_p2p(const int* uu_ptr, const int* uu_col, const float* uu_val, const float* diag, int m, int l, int row_lo,
                         int row_hi, const gll_peers* peers, unsigned epoch, const int* ctrl, void* workspace,
                         size_t workspace_bytes, void* stream);
int gll_cg_rows_update_p2p(const float* diag, int m, int l, int row_lo, int row_hi, int iter, int max_iter, float tol, float* x,
                           const gll_peers* peers, unsigned epoch, int* ctrl, float* resid_out, void* workspace,
                           size_t workspace_bytes, void* stream);
/* m x lp fp32 -> m x l float64/fp32 (GLL.py:66) and m x l float64/fp32 grad_output -> m x lp fp32 (GLL.py:90). */
int gll_unpack_pred(const float* u, int m, int l, void* pred, int pred_is_f64, void* stream);
int gll_pack_grad(const void* grad_out, int grad_is_f64, int m, int l, float* rhs, void* stream);

/* The step in front of the layer in every caller: F.normalize(feat, dim=1) (networks/BuildNet.py:101), and its backward.
 * Xn = X / max(|X_row|, eps) (eps = 1e-12 in PyTorch); inv_norm[n] is kept for the backward (sign bit set for rows that
 * hit the clamp); dX = (dXn - Xn <Xn, dXn>) * inv_norm.  X, Xn, dXn, dX: n x d fp32 row-major. */
int gll_normalize_rows(const float* X, int n, int d, float eps, float* Xn, float* inv_norm, void* stream);
int gll_normalize_rows_backward(const float* Xn, const float* inv_norm, const float* dXn, int n, int d, float* dX, void* stream);

/* r = b - A x in fp64: A in CSR (diagonal included, int32 indices, fp64 values, m x m), x, b, r dense m x l row-major fp64.
 * The iterative-refinement residual of the stable_conjgrad wrapper (GLL.py:247-276, tol = 1e-10). */
int gll_csr_residual_f64(const int* ptr, const int* col, const double* val, const double* x, const double* b, int m, int l,
                         double* r, void* stream);

/* The loss every caller of the layer applies to its output (custom_ce_loss, losses.py:128-136; also pasted at
 * train_and_adversarial.py:458 and adversarial.py:453): loss = -sum_i log(pred[i, targets[i]] + 1e-8) / m, and in the same
 * launch d loss / d pred (m x l, same dtype as pred).  pred: m x l float64 (pred_is_f64 != 0) or fp32; targets: m int64;
 * loss_out: one element of pred's dtype.  status (optional, device int): GLL_STATUS_NONFINITE is or-ed in when a target
 * is outside [0, l). */
size_t gll_ce_loss_workspace_bytes(int m);  /* 0 for m <= 4096 (one CTA writes the loss directly) */
int gll_ce_loss(const void* pred, int pred_is_f64, const long long* targets, int m, int l, void* loss_out, void* grad_out,
                int* status, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused drivers: what LaplaceLearningSparseHard.forward / .backward call (GLL.py:13-73, 75-177).
 * `state` is a buffer of gll_state_layout(...).total bytes that must stay alive (and untouched) between the
 * two calls; `workspace` may be reused by anybody in between.
 * pred_out: m x l, float64 when pred_is_f64 != 0 (the reference returns float64, GLL.py:66) else fp32.
 * grad_out: m x l, float64 when grad_is_f64 != 0 else fp32.  dX: n x d fp32 (GLL.py:154,159).
 * ------------------------------------------------------------------------------------------- */
int gll_forward(const float* X, const float* Y, int n, int d, int k, int l, int k_lab, int eps_auto,
                float eps_fixed, float tau, float cg_tol, int cg_max_iter, void* state, void* pred_out,
                int pred_is_f64, void* workspace, size_t workspace_bytes, void* stream);

int gll_backward(const float* X, const void* grad_out, int grad_is_f64, int n, int d, int k, int l, int k_lab,
                 int eps_auto, float cg_tol, int cg_max_iter, void* state, float* dX, void* workspace,
                 size_t workspace_bytes, void* stream);
/* The same with a device scalar multiplied into grad_out (scale == NULL: 1): the upstream gradient of a loss head whose
 * d loss / d Pred is grad_out (custom_ce_loss fused behind the layer, losses.py:128-136 after FullySup.py:156-158); no host read. */
int gll_backward_scaled(const float* X, const void* grad_out, int grad_is_f64, const void* scale, int scale_is_f64, int n, int d,
                        int k, int l, int k_lab, int eps_auto, float cg_tol, int cg_max_iter, void* state, float* dX,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Batched forward of B independent graphs of the same shape (LaplaceLearningSparseHardBatched): X is B x n x d and Y is
 * B x k_lab x l, each graph's labeled rows first.  The B graphs are ONE block-diagonal graph whose rows are ordered labeled
 * first: all graphs' labeled rows (graph-major), then all graphs' unlabeled rows (graph-major), each graph's rows in their
 * own order.  The kNN search runs per graph (gll_knn_segments); graph, weights and the CG are gll_forward's stages on the
 * union, so state has the layout of gll_state_layout(B n, k, l, B k_lab), its kNN lists, CSR, eps, kappa, W and degrees are
 * per graph bit-identical to gll_forward's, and pred_out (B*(n - k_lab)) x l is graph-major: a (B, m, l) tensor.  One
 * multi-RHS CG solves all graphs (step lengths shared, each class column stops when its residual over all graphs is
 * <= cg_tol, which bounds every graph's), so pred matches per-graph calls to the solver tolerance, not bit for bit, for B > 1.
 * The backward is gll_backward_scaled(Xg, ..., B n, d, k, l, B k_lab, ...) on Xg = X in labeled-first order. */
size_t gll_batched_workspace_bytes(int B, int n, int d, int k, int l, int k_lab);
int gll_forward_batched(const float* X, const float* Y, int B, int n, int d, int k, int l, int k_lab, int eps_auto,
                        float eps_fixed, float tau, float cg_tol, int cg_max_iter, void* state, void* pred_out,
                        int pred_is_f64, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Laplace-learning evaluation, the reference's utils.laplace (utils.py:570-593) as test_GL_NP calls it (utils.py:637-660):
 * one graph over all n rows (labeled rows first), the unlabeled block solved to the reference's stop rule, argmax labels.
 *   Graph: gll_forward's stages with this k (2 <= k <= 64; n >= 256 when k > 33), eps_auto / eps_fixed as there.
 *   System: L = D - W from the stored fp32 W, evaluated in fp64, with D = ROW sums of W (the reference's csgraph.laplacian
 *   takes column sums; W_ij and W_ji may differ in the last fp32 bit, so the two agree to ~1e-7 relative).
 *   Solve (L_uu + tau I) x = -L_ul Y: fp32 Jacobi-CG, then GLL_LAPLACE_ROUNDS rounds of fp64 residual + fp32 correction solve,
 *   stopping when every class column has ||M (b - A x)||_2 <= tol, M = diag(A + 1e-10)^(-1/2) -- the residual of the
 *   reference's stable_conjgrad on the Jacobi-scaled system.  Rounds after convergence cost two launches and no iterations.
 *   Outputs: pred m x l fp64 (m = n - k_lab), labels[m] int64 = first maximal column; with targets (m int64, may be NULL)
 *   correct_out (one int64, may be NULL) = #{i : targets[i] >= 0 and labels[i] == targets[i]}.
 *   info: GLL_INFO_WORDS int32 (device); GLL_STATUS_CG_NOT_CONVERGED when tol is unmet after the last round.
 *   workspace: gll_laplace_eval_workspace_bytes(...) bytes (it also holds the graph state).  Nothing syncs with the host. */
size_t gll_laplace_eval_workspace_bytes(int n, int d, int k, int l, int k_lab);
int gll_laplace_eval(const float* X, const float* Y, int n, int d, int k, int l, int k_lab, int eps_auto, float eps_fixed,
                     float tau, double tol, int cg_max_iter, double* pred, long long* labels, const long long* targets,
                     long long* correct_out, int* info, void* workspace, size_t workspace_bytes, void* stream);

/* gll_laplace_eval over B independent graphs of the same shape: X is B x n x d and Y is B x k_lab x l, each graph's labeled
 * rows first.  As gll_forward_batched, the graphs are one block-diagonal graph in labeled-first order: the kNN search runs per
 * graph (gll_knn_segments, so every graph's lists, CSR and W are bit-identical to a per-graph call), then the stages, the
 * solves and the refinement of gll_laplace_eval run on the union.  The stop rule is per graph: the refinement stops when every
 * class column of EVERY graph has ||M (b - A x)||_2 <= tol over that graph's rows; while one graph is above tol all graphs get
 * corrections.  The CG step lengths are shared by the graphs, so pred matches per-graph gll_laplace_eval calls to solver
 * accuracy, not bit for bit; B = 1 is bit-identical to gll_laplace_eval.
 *   Sizes: B >= 1, B n < 2^31, 2 <= k <= 64, k <= n, B n >= 256 when k > 33, 1 <= k_lab < n, l >= 1, tol > 0, cg_max_iter >= 1.
 *   Outputs: pred (B m) x l fp64 and labels[B m] int64 are graph-major ((B, m, l) and (B, m), m = n - k_lab); targets
 *   (B m int64, may be NULL) line up with them; correct_out (B int64, may be NULL) counts hits per graph; resid_out (B fp64,
 *   may be NULL) = per graph the largest column norm of the last round (GLL_INFO_LAPLACE_RESID's meaning, per graph).
 *   info: as gll_laplace_eval, the residual slots holding the maximum over graphs and the iteration counts those of the whole
 *   batch.  Bad arguments return GLL_ERR_ARG before any CUDA call; the workspace query returns 0 for them.  Nothing syncs with
 *   the host, so the call can be captured in a CUDA graph. */
size_t gll_laplace_eval_batched_workspace_bytes(int B, int n, int d, int k, int l, int k_lab);
int gll_laplace_eval_batched(const float* X, const float* Y, int B, int n, int d, int k, int l, int k_lab, int eps_auto,
                             float eps_fixed, float tau, double tol, int cg_max_iter, double* pred, long long* labels,
                             const long long* targets, long long* correct_out, double* resid_out, int* info,
                             void* workspace, size_t workspace_bytes, void* stream);

/* T trials of gll_laplace_eval on ONE set of features: trial t labels the k_lab rows train_idx[t] (T x k_lab, int64 when
 * idx_is_i64, else int32; device) with Y[t] (T x k_lab x l fp32) and solves the other n - k_lab rows.  X (n x d) is in any row
 * order.  The graph (kNN, CSR, eps, W, degrees) is built once on X in natural order, as gll_laplace_eval's stages with no labeled
 * rows; trial t's result is gll_laplace_eval on X[perm_t], perm_t = [train_idx[t], the other rows in natural order], mapped back
 * to natural order.  Without exact distance ties the graph is the permuted graph of every trial; on exact ties the index
 * tie-break of the kNN search follows natural order, not perm_t.
 *   Solve: all T l class columns against one full-graph system A = D + tau I - W; trial t's labeled rows are masked out of its
 *   columns (A p is zeroed there), each column keeps its own CG step lengths, and the fp64 refinement stops when every class column
 *   of every valid trial has ||M (b - A x)||_2 <= tol over that trial's unlabeled rows (M, D as gll_laplace_eval).
 *   Invalid trials: a train_idx row with an index outside [0, n) or a repeated index never causes an out-of-bounds access; the
 *   trial gets a zero right-hand side (it neither stops nor slows the others), pred NaN, labels -1, correct -1, resid NaN, and
 *   GLL_STATUS_BAD_INDEX is set.  The other trials are unaffected.
 *   Sizes: n >= 2, T >= 1, n T lpad < 2^31 (lpad = gll_padded_classes(l)), T l <= 2097120, 2 <= k <= 64, k <= n, n >= 256
 *   when k > 33, 1 <= k_lab < n, l >= 1, d >= 1, tol > 0, cg_max_iter >= 1.
 *   Outputs: pred T x n x l fp64 and labels T x n int64 (a row labeled in trial t gets its label row and that row's argmax);
 *   targets (n int64, may be NULL; negative = not scored); correct_out (T int64, may be NULL) counts per trial the rows that are
 *   not labeled in it and whose label equals their target; resid_out (T fp64, may be NULL) = per trial the largest column norm of
 *   the last round.  info: as gll_laplace_eval, residual slots holding the maximum over valid trials.  Bad arguments return
 *   GLL_ERR_ARG before any CUDA call; the workspace query returns 0 for them.  Nothing syncs with the host and nothing is copied,
 *   so the call can be captured in a CUDA graph. */
size_t gll_laplace_eval_trials_workspace_bytes(int n, int d, int k, int l, int T, int k_lab);
int gll_laplace_eval_trials(const float* X, int n, int d, int k, const void* train_idx, int idx_is_i64, const float* Y, int T,
                            int k_lab, int l, int eps_auto, float eps_fixed, float tau, double tol, int cg_max_iter, double* pred,
                            long long* labels, const long long* targets, long long* correct_out, double* resid_out, int* info,
                            void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GLL_B200_H */
