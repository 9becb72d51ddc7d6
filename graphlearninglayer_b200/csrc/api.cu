// C ABI of libgll_b200.so (see include/gll_b200.h) and the fused forward / backward drivers.
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <vector>

#include "cg_common.cuh"
#include "common.cuh"

namespace gll {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

const DeviceInfo& device_info() {
  static thread_local DeviceInfo cache[64];
  static thread_local bool have[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (!have[dev]) {
    DeviceInfo di;
    di.device = dev;
    di.sms = 148;
    di.max_smem_optin = 227 * 1024;
    cudaDeviceGetAttribute(&di.sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&di.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (di.sms <= 0) di.sms = 148;
    cache[dev] = di;
    have[dev] = true;
  }
  return cache[dev];
}

cudaError_t set_max_dynamic_smem_once(const void* func, int bytes) {
  struct Key {
    const void* f;
    int dev, bytes;
  };
  static std::mutex mu;
  static std::vector<Key> done;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lk(mu);
  for (const Key& k : done)
    if (k.f == func && k.dev == dev && k.bytes >= bytes) return cudaSuccess;
  e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) done.push_back(Key{func, dev, bytes});
  return e;
}

// ------------------------------------------------------------------------------------------------ profiling
namespace {
struct ProfRec {
  int id;
  cudaEvent_t e0, e1;
};
std::mutex g_prof_mu;
std::vector<ProfRec*> g_prof_recs;
std::atomic<int> g_prof_on{0};
std::atomic<long long> g_launches[KID_COUNT];
const char* const g_kernel_names[KID_COUNT] = {
    "sqnorm", "knn_gram_topk_simt", "knn_gram_topk_tcgen05", "knn_rerank", "knn_fallback", "graph_build", "edge_weights",
    "cg_persistent", "pack_unpack", "edge_grad", "row_gather", "convert", "cg_rows", "laplace_refine", "laplace_finish",
    "knn_segment_setup", "batch_reorder", "laplace_trials_setup"};
}  // namespace

ProfScope::ProfScope(int id_, cudaStream_t st_) : id(id_), st(st_), slot(nullptr) {
  g_launches[id].fetch_add(1, std::memory_order_relaxed);
  if (g_prof_on.load(std::memory_order_relaxed)) {
    ProfRec* r = new ProfRec;
    r->id = id;
    cudaEventCreate(&r->e0);
    cudaEventCreate(&r->e1);
    cudaEventRecord(r->e0, st);
    slot = r;
  }
}
ProfScope::~ProfScope() {
  if (slot) {
    ProfRec* r = (ProfRec*)slot;
    cudaEventRecord(r->e1, st);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof_recs.push_back(r);
  }
}

namespace {

// rhs = grad_output padded to lp class columns (fp32); optionally also wt[0 : zero_count] = 0 (the labeled rows of the
// padded adjoint solution, GLL.py:104) so that the backward needs no separate memset
__global__ void pack_grad_kernel(const void* __restrict__ g, int is_f64, int m, int l, int lp, float* __restrict__ rhs,
                                 float* __restrict__ zero_ptr, long long zero_count, const void* __restrict__ scale, int scale_f64) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (long long z = t; z < zero_count; z += (long long)gridDim.x * blockDim.x) zero_ptr[z] = 0.f;
  if (t >= (long long)m * lp) return;
  int r = (int)(t / lp), c = (int)(t % lp);
  const double sc = (scale == nullptr) ? 1.0 : (scale_f64 ? *(const double*)scale : (double)*(const float*)scale);
  float v = 0.f;
  if (c < l) v = is_f64 ? (float)(sc * ((const double*)g)[(size_t)r * l + c]) : (float)(sc * (double)((const float*)g)[(size_t)r * l + c]);
  rhs[t] = v;
}

// custom_ce_loss (losses.py:128-136): loss = -sum_i log(p[i, t_i] + 1e-8) / m and, in the same pass, its gradient
// d loss / d p[i, c] = -[c == t_i] / (m (p[i, t_i] + 1e-8)).  Fixed summation order: per-CTA sums in CTA order.
// One CTA writes the loss directly (minibatch sizes); with several CTAs each writes its partial sum and
// ce_loss_finish_kernel adds them.
template <typename T>
__global__ void __launch_bounds__(1024) ce_loss_kernel(const T* __restrict__ p, const long long* __restrict__ tgt, int m, int l,
                                                        T* __restrict__ loss, T* __restrict__ grad, double* __restrict__ partial,
                                                        int* __restrict__ status) {
  __shared__ double part[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double acc = 0.0;
  const double inv_m = 1.0 / (double)m;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
    const long long t = tgt[i];
    const bool ok = t >= 0 && t < l;
    if (!ok && status) atomicOr(status, GLL_STATUS_NONFINITE);
    const double q = ok ? (double)p[(size_t)i * l + t] + 1e-8 : 1.0;
    acc += log(q);
    for (int c = 0; c < l; ++c) grad[(size_t)i * l + c] = (T)((ok && c == t) ? -inv_m / q : 0.0);
  }
  acc = warp_sum(acc);
  if (lane == 0) part[warp] = acc;
  __syncthreads();
  if (warp == 0) {
    double v = (lane < (int)(blockDim.x >> 5)) ? part[lane] : 0.0;
    v = warp_sum(v);
    if (lane == 0) {
      if (gridDim.x == 1)
        *loss = (T)(-v * inv_m);
      else
        partial[blockIdx.x] = v;
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(32) ce_loss_finish_kernel(const double* __restrict__ partial, int blocks, int m, T* __restrict__ loss) {
  double v = 0.0;
  for (int b = threadIdx.x; b < blocks; b += 32) v += partial[b];
  v = warp_sum(v);
  if (threadIdx.x == 0) *loss = (T)(-v / (double)m);
}

// F.normalize(feat, dim=1) (networks/BuildNet.py:101: every caller feeds the layer L2-normalised rows) and its backward,
// one warp per row each:  xn = x / max(|x|, eps);  dx = (dxn - xn <xn, dxn>) / |x|   (dx = dxn / eps where |x| <= eps).
__global__ void __launch_bounds__(256)
normalize_rows_kernel(const float* __restrict__ X, int n, int d, float eps, float* __restrict__ Xn, float* __restrict__ inv_norm) {
  const int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (row >= n) return;
  const float* x = X + (size_t)row * d;
  double s = 0.0;
  for (int c = lane; c < d; c += 32) {
    const double v = (double)__ldg(x + c);
    s += v * v;
  }
  s = warp_sum(s);
  const float nrm = (float)sqrt(s);
  const float inv = 1.f / fmaxf(nrm, eps);
  for (int c = lane; c < d; c += 32) Xn[(size_t)row * d + c] = __ldg(x + c) * inv;
  if (lane == 0) inv_norm[row] = (nrm > eps) ? inv : -inv;  // sign bit marks the clamped rows (no projection in the backward)
}

__global__ void __launch_bounds__(256)
normalize_rows_backward_kernel(const float* __restrict__ Xn, const float* __restrict__ inv_norm, const float* __restrict__ dXn, int n,
                               int d, float* __restrict__ dX) {
  const int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (row >= n) return;
  const float* xn = Xn + (size_t)row * d;
  const float* g = dXn + (size_t)row * d;
  const float iv = inv_norm[row];
  double dot = 0.0;
  if (iv > 0.f) {
    for (int c = lane; c < d; c += 32) dot += (double)__ldg(xn + c) * (double)__ldg(g + c);
    dot = warp_sum(dot);
  }
  const float dt = (float)dot, inv = fabsf(iv);
  for (int c = lane; c < d; c += 32) dX[(size_t)row * d + c] = (__ldg(g + c) - __ldg(xn + c) * dt) * inv;
}

// r = b - A x in fp64 (CSR with the diagonal included, int32 indices, m x l dense row-major): the refinement residual of
// the stable_conjgrad wrapper (GLL.py:247-276 asks for ||b - A x|| <= 1e-10, below what the fp32 solver alone reaches).
// One thread per (row, class column): lanes run along the contiguous class index.
__global__ void __launch_bounds__(256)
csr_residual_f64_kernel(const int* __restrict__ ptr, const int* __restrict__ col, const double* __restrict__ val,
                        const double* __restrict__ x, const double* __restrict__ b, int m, int l, double* __restrict__ r) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)m * l) return;
  const int i = (int)(t / l), c = (int)(t - (long long)i * l);
  double acc = b[t];
  const int e1 = ptr[i + 1];
  for (int e = ptr[i]; e < e1; ++e) acc = fma(-val[e], x[(size_t)col[e] * l + c], acc);
  r[t] = acc;
}

__global__ void unpack_pred_kernel(const float* __restrict__ u, int m, int l, int lp, void* __restrict__ pred, int is_f64) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)m * l) return;
  int r = (int)(t / l), c = (int)(t % l);
  float v = u[(size_t)r * lp + c];
  if (is_f64)
    ((double*)pred)[t] = (double)v;
  else
    ((float*)pred)[t] = v;
}

// Batched layer: natural order (graph b, row t) -> the block-diagonal graph's order, all graphs' labeled rows first, then all
// graphs' unlabeled rows, each graph's rows in their own order
__device__ __forceinline__ int labeled_first_row(int r, int n, int k_lab, int B) {
  const int b = r / n, t = r - b * n;
  return (t < k_lab) ? b * k_lab + t : B * k_lab + b * (n - k_lab) + (t - k_lab);
}

// kNN lists of the stacked graphs in natural order -> rows and indices in labeled-first order
__global__ void knn_to_labeled_first_kernel(const int* __restrict__ idx_in, const float* __restrict__ dist_in, int B, int n, int k,
                                            int k_lab, int* __restrict__ idx_out, float* __restrict__ dist_out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)B * n * k) return;
  const int r = (int)(t / k), s = (int)(t - (long long)r * k);
  const size_t o = (size_t)labeled_first_row(r, n, k_lab, B) * k + s;
  idx_out[o] = labeled_first_row(idx_in[t], n, k_lab, B);
  dist_out[o] = dist_in[t];
}

__global__ void pack_columns_kernel(const float* __restrict__ src, int rows, int lp_src, int c0, int cnt, float* __restrict__ dst,
                                    int lp_dst) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)rows * lp_dst) return;
  int r = (int)(t / lp_dst), c = (int)(t % lp_dst);
  dst[t] = (c < cnt) ? src[(size_t)r * lp_src + c0 + c] : 0.f;
}

__global__ void unpack_columns_kernel(const float* __restrict__ src, int rows, int lp_src, int c0, int cnt, float* __restrict__ dst,
                                      int lp_dst) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)rows * cnt) return;
  int r = (int)(t / cnt), c = (int)(t % cnt);
  dst[(size_t)r * lp_dst + c0 + c] = src[(size_t)r * lp_src + c];
}

}  // namespace

int pack_columns(const float* src, int rows, int lp_src, int c0, int cnt, float* dst, int lp_dst, cudaStream_t st) {
  GLL_PROF(KID_PACK, st);
  pack_columns_kernel<<<ceil_div((long long)rows * lp_dst, 256), 256, 0, st>>>(src, rows, lp_src, c0, cnt, dst, lp_dst);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

int unpack_columns(const float* src, int rows, int lp_src, int c0, int cnt, float* dst, int lp_dst, cudaStream_t st) {
  if (cnt <= 0) return GLL_OK;
  GLL_PROF(KID_PACK, st);
  unpack_columns_kernel<<<ceil_div((long long)rows * cnt, 256), 256, 0, st>>>(src, rows, lp_src, c0, cnt, dst, lp_dst);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

int pack_grad(const void* g, int is_f64, int m, int l, int lp, float* rhs, cudaStream_t st, float* zero_ptr, long long zero_count,
              const void* scale, int scale_f64) {
  GLL_PROF(KID_PACK, st);
  pack_grad_kernel<<<ceil_div((long long)m * lp, 256), 256, 0, st>>>(g, is_f64, m, l, lp, rhs, zero_ptr, zero_count, scale, scale_f64);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

int unpack_pred(const float* ut_u, int m, int l, int lp, void* pred, int is_f64, cudaStream_t st) {
  GLL_PROF(KID_PACK, st);
  unpack_pred_kernel<<<ceil_div((long long)m * l, 256), 256, 0, st>>>(ut_u, m, l, lp, pred, is_f64);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

static int make_layout(int n, int k, int l, int k_lab, gll_layout* L) {
  if (!L || n < 1 || k < 2 || l < 1 || k_lab < 0 || k_lab >= n) return GLL_ERR_ARG;
  const size_t emax = gll_max_edges(n, k), lp = (size_t)padded_classes(l), m = (size_t)(n - k_lab);
  size_t off = 0;
  auto put = [&](size_t bytes) {
    size_t o = align_up(off, 256);
    off = o + bytes;
    return o;
  };
  L->knn_idx = put(4 * (size_t)n * k);
  L->knn_dist = put(4 * (size_t)n * k);
  L->row_ptr = put(4 * ((size_t)n + 1));
  L->col = put(4 * emax);
  L->dist = put(4 * emax);
  L->w = put(4 * emax);
  L->gv = put(4 * emax);
  L->eps = put(4 * (size_t)n);
  L->kappa = put(4 * (size_t)n);
  L->deg = put(4 * (size_t)n);
  L->bvec = put(4 * (size_t)n);
  L->uu_ptr = put(4 * (m + 1));
  L->uu_col = put(4 * emax);
  L->uu_val = put(4 * emax);
  L->diag = put(4 * m);
  L->rhs = put(4 * m * lp);
  L->ut = put(4 * (size_t)n * lp);
  L->wt = put(4 * (size_t)n * lp);
  L->info = put(4 * GLL_INFO_WORDS);
  L->total = align_up(off, 256);
  return GLL_OK;
}

// expected off-diagonal entries per row of L_uu: the solver's sparsity hint in gll_forward / gll_backward.  evalcache._uu_hint
// repeats this float32 arithmetic bit for bit so that BaseSetEvaluator runs the same solver kernel.
static float uu_degree_hint(int n, int k, int m) { return 1.2f * (float)(k - 1) * (float)m / (float)n; }

GraphBufs graph_bufs(const gll_layout& L, void* state) {
  char* S = (char*)state;
  GraphBufs B;
  B.knn_idx = (int*)(S + L.knn_idx);
  B.knn_dist = (float*)(S + L.knn_dist);
  B.row_ptr = (int*)(S + L.row_ptr);
  B.col = (int*)(S + L.col);
  B.dist = (float*)(S + L.dist);
  B.w = (float*)(S + L.w);
  B.gv = (float*)(S + L.gv);
  B.eps = (float*)(S + L.eps);
  B.kappa = (int*)(S + L.kappa);
  B.deg = (float*)(S + L.deg);
  B.bvec = (float*)(S + L.bvec);
  B.uu_ptr = (int*)(S + L.uu_ptr);
  B.uu_col = (int*)(S + L.uu_col);
  B.uu_val = (float*)(S + L.uu_val);
  B.diag = (float*)(S + L.diag);
  B.rhs = (float*)(S + L.rhs);
  B.ut = (float*)(S + L.ut);
  B.wt = (float*)(S + L.wt);
  B.info = (int*)(S + L.info);
  return B;
}

}  // namespace gll

using namespace gll;

extern "C" {

const char* gll_last_error(void) { return g_err; }
int gll_version(void) { return 100; }
int gll_device_sm_count(void) { return device_info().sms; }
int gll_padded_classes(int l) { return padded_classes(l); }
size_t gll_max_edges(int n, int k) { return (size_t)2 * (size_t)n * (size_t)(k - 1); }

int gll_kernel_count(void) { return KID_COUNT; }
const char* gll_kernel_name(int id) { return (id >= 0 && id < KID_COUNT) ? g_kernel_names[id] : ""; }
long long gll_launch_count(int id) {
  if (id >= 0 && id < KID_COUNT) return g_launches[id].load();
  long long t = 0;
  for (int i = 0; i < KID_COUNT; ++i) t += g_launches[i].load();
  return t;
}
void gll_debug_cg_trace(void* device_buf) { cg_set_trace(device_buf); }
void gll_debug_knn_trace(void* device_buf) { knn_tc_set_trace(device_buf); }
void gll_profile_enable(int on) { g_prof_on.store(on ? 1 : 0); }
int gll_profile_collect(double* ms_sum, long long* count) {
  std::vector<ProfRec*> recs;
  {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    recs.swap(g_prof_recs);
  }
  for (int i = 0; i < KID_COUNT; ++i) {
    if (ms_sum) ms_sum[i] = 0.0;
    if (count) count[i] = 0;
  }
  int rc = GLL_OK;
  for (ProfRec* r : recs) {
    float ms = 0.f;
    if (cudaEventSynchronize(r->e1) != cudaSuccess || cudaEventElapsedTime(&ms, r->e0, r->e1) != cudaSuccess) {
      set_error("gll_profile_collect: event query failed");
      rc = GLL_ERR_CUDA;
    } else {
      if (ms_sum) ms_sum[r->id] += (double)ms;
      if (count) count[r->id] += 1;
    }
    cudaEventDestroy(r->e0);
    cudaEventDestroy(r->e1);
    delete r;
  }
  return rc;
}

int gll_state_layout(int n, int k, int l, int k_lab, gll_layout* out) {
  int rc = make_layout(n, k, l, k_lab, out);
  if (rc) set_error("gll_state_layout: bad sizes n=%d k=%d l=%d k_lab=%d", n, k, l, k_lab);
  return rc;
}

size_t gll_knn_workspace_bytes(int n, int d, int k) { return knn_ws_bytes(n, d, k, 0, n); }
size_t gll_knn_rows_workspace_bytes(int n, int d, int k, int row_begin, int row_end) {
  return knn_ws_bytes(n, d, k, row_begin, row_end);
}
size_t gll_graph_workspace_bytes(int n, int k) { return graph_ws_bytes(n, k); }
size_t gll_weights_workspace_bytes(int n, int k) { return weights_ws_bytes(n, k); }
size_t gll_cg_workspace_bytes(int m, int l) { return cg_ws_bytes(m, l); }

size_t gll_workspace_bytes(int n, int d, int k, int l, int k_lab) {
  size_t b = knn_ws_bytes(n, d, k, 0, n);
  size_t t = graph_weights_ws_bytes(n, k);
  if (t > b) b = t;
  t = cg_ws_bytes(n - k_lab > 0 ? n - k_lab : 1, l);
  if (t > b) b = t;
  return b;
}

int gll_knn(const float* X, int n, int d, int k, int* knn_idx, float* knn_dist, int* info, void* workspace,
            size_t workspace_bytes, void* stream) {
  return knn_run(X, n, d, k, 0, n, knn_idx, knn_dist, info, workspace, workspace_bytes, (cudaStream_t)stream);
}

size_t gll_base_cache_bytes(int n_base) { return knn_base_cache_bytes(n_base); }
size_t gll_base_cache_workspace_bytes(int n_base, int d) { return knn_ws_bytes(n_base, d, 25, 0, n_base); }
int gll_base_cache_build(const float* Xbase, int n_base, int d, void* cache, void* workspace, size_t workspace_bytes, void* stream) {
  return knn_base_cache_build(Xbase, n_base, d, cache, workspace, workspace_bytes, (cudaStream_t)stream);
}
size_t gll_knn_cached_workspace_bytes(int n, int d, int k, int n_base) { return knn_cached_ws_bytes(n, d, k, n_base); }
int gll_knn_cached(const float* X, int n, int d, int k, int n_base, const void* cache, int* knn_idx, float* knn_dist, int* info,
                   void* workspace, size_t workspace_bytes, void* stream) {
  return knn_run_cached(X, n, d, k, n_base, cache, knn_idx, knn_dist, info, workspace, workspace_bytes, (cudaStream_t)stream);
}

int gll_debug_gram_tile(const float* X, int n, int d, int row_tile, int col_tile, float* acc_out, float* rscale_out, void* workspace,
                        size_t workspace_bytes, void* stream) {
  return knn_debug_gram_tile(X, n, d, row_tile, col_tile, acc_out, rscale_out, workspace, workspace_bytes, (cudaStream_t)stream);
}

int gll_knn_rows(const float* X, int n, int d, int k, int row_begin, int row_end, int* knn_idx, float* knn_dist, int* info,
                 void* workspace, size_t workspace_bytes, void* stream) {
  return knn_run(X, n, d, k, row_begin, row_end, knn_idx, knn_dist, info, workspace, workspace_bytes, (cudaStream_t)stream);
}

int gll_graph_build(const int* knn_idx, const float* knn_dist, int n, int k, int* row_ptr, int* col, float* dist, int* info,
                    void* workspace, size_t workspace_bytes, void* stream) {
  GraphBufs B = {};
  B.knn_idx = const_cast<int*>(knn_idx);  // inputs: only read
  B.knn_dist = const_cast<float*>(knn_dist);
  B.row_ptr = row_ptr;
  B.col = col;
  B.dist = dist;
  B.info = info;
  return graph_stages_run(B, nullptr, n, k, 0, 0, 0, 0.f, 0.f, /*phases*/ 0, 4, workspace, workspace_bytes, (cudaStream_t)stream);
}

int gll_edge_weights(const int* knn_idx, const float* knn_dist, const int* row_ptr, const int* col, const float* dist,
                     const float* Y, int n, int k, int l, int k_lab, int eps_auto, float eps_fixed, float tau, float* eps,
                     int* kappa, float* w, float* deg, int* uu_ptr, int* uu_col, float* uu_val, float* diag, float* rhs,
                     float* ut, int* info, void* workspace, size_t workspace_bytes, void* stream) {
  GraphBufs B = {};
  B.knn_idx = const_cast<int*>(knn_idx);  // inputs: only read
  B.knn_dist = const_cast<float*>(knn_dist);
  B.row_ptr = const_cast<int*>(row_ptr);
  B.col = const_cast<int*>(col);
  B.dist = const_cast<float*>(dist);
  B.eps = eps;
  B.kappa = kappa;
  B.w = w;
  B.deg = deg;
  B.uu_ptr = uu_ptr;
  B.uu_col = uu_col;
  B.uu_val = uu_val;
  B.diag = diag;
  B.rhs = rhs;
  B.ut = ut;
  B.info = info;
  return graph_stages_run(B, Y, n, k, l, k_lab, eps_auto, eps_fixed, tau, /*phases*/ 3, 6, workspace, workspace_bytes, (cudaStream_t)stream);
}

int gll_cg_solve(const int* uu_ptr, const int* uu_col, const float* uu_val, const float* diag, const float* rhs, int m, int l,
                 float tol, int max_iter, float* x, int* iters_out, float* resid_out, int* status_out, void* workspace,
                 size_t workspace_bytes, void* stream) {
  return gll_cg_solve_hint(uu_ptr, uu_col, uu_val, diag, rhs, m, l, tol, max_iter, x, iters_out, resid_out, status_out, workspace,
                           workspace_bytes, stream, 0.f);
}

int gll_cg_solve_hint(const int* uu_ptr, const int* uu_col, const float* uu_val, const float* diag, const float* rhs, int m, int l,
                      float tol, int max_iter, float* x, int* iters_out, float* resid_out, int* status_out, void* workspace,
                      size_t workspace_bytes, void* stream, float uu_degree_hint) {
  CgSolve S{};
  S.ptr = uu_ptr;
  S.col = uu_col;
  S.val = uu_val;
  S.diag = diag;
  S.m = m;
  S.rhs = rhs;
  S.x = x;
  S.l = l;
  S.tol = tol;
  S.max_iter = max_iter;
  S.iters_out = iters_out;
  S.resid_out = resid_out;
  S.status_out = status_out;
  S.uu_degree_hint = uu_degree_hint;
  return cg_run(S, workspace, workspace_bytes, (cudaStream_t)stream);
}

int gll_cg_kernel(int m, int l, float uu_degree_hint) {
  GLL_REQUIRE(m >= 1 && l >= 1 && l <= 128, "need m >= 1 and 1 <= l <= 128");
  return cg_pick(m, padded_classes(l), uu_degree_hint, false);
}

int gll_backward_edges(const float* X, int n, int d, int l, int k_lab, int eps_auto, const int* row_ptr, const int* col,
                       const float* dist, const float* w, const float* eps, const int* kappa, const float* ut,
                       const float* wt, float* gv, float* bvec, float* dX, void* stream) {
  return gll_backward_edges_rows(X, n, d, l, k_lab, eps_auto, row_ptr, col, dist, w, eps, kappa, ut, wt, gv, bvec, dX, 0, n, 3,
                                 stream);
}

int gll_backward_edges_rows(const float* X, int n, int d, int l, int k_lab, int eps_auto, const int* row_ptr, const int* col,
                            const float* dist, const float* w, const float* eps, const int* kappa, const float* ut,
                            const float* wt, float* gv, float* bvec, float* dX, int row_begin, int row_end, int phases,
                            void* stream) {
  GraphBufs B = {};
  B.row_ptr = const_cast<int*>(row_ptr);  // inputs: only read
  B.col = const_cast<int*>(col);
  B.dist = const_cast<float*>(dist);
  B.w = const_cast<float*>(w);
  B.eps = const_cast<float*>(eps);
  B.kappa = const_cast<int*>(kappa);
  B.ut = const_cast<float*>(ut);
  B.wt = const_cast<float*>(wt);
  B.gv = gv;
  B.bvec = bvec;
  return backward_edges_run(X, n, d, l, k_lab, eps_auto, B, dX, row_begin, row_end, phases, (cudaStream_t)stream);
}

size_t gll_cg_rows_workspace_bytes(int rows_local, int l) { return cg_rows_ws_bytes(rows_local, l); }

int gll_cg_rows_init(const float* diag, const float* rhs, int m, int l, int row_lo, int row_hi, float* x, float* u_full,
                     void* workspace, size_t workspace_bytes, void* stream) {
  return cg_rows_init(diag, rhs, m, l, row_lo, row_hi, x, u_full, workspace, workspace_bytes, nullptr, 0u, (cudaStream_t)stream);
}

int gll_cg_rows_spmv(const int* uu_ptr, const int* uu_col, const float* uu_val, const float* diag, int m, int l, int row_lo,
                     int row_hi, const float* u_full, double* sums, void* workspace, size_t workspace_bytes, void* stream) {
  return cg_rows_spmv(uu_ptr, uu_col, uu_val, diag, m, l, row_lo, row_hi, u_full, sums, workspace, workspace_bytes, nullptr, 0u,
                      nullptr, (cudaStream_t)stream);
}

int gll_cg_rows_update(const float* diag, int m, int l, int row_lo, int row_hi, const double* sums, int iter, int max_iter,
                       float tol, float* x, float* u_full, int* ctrl, float* resid_out, void* workspace, size_t workspace_bytes,
                       void* stream) {
  return cg_rows_update(diag, m, l, row_lo, row_hi, sums, iter, max_iter, tol, x, u_full, ctrl, resid_out, workspace,
                        workspace_bytes, nullptr, 0u, (cudaStream_t)stream);
}

size_t gll_ce_loss_workspace_bytes(int m) { return (m <= 4096) ? 0 : sizeof(double) * 1024; }

int gll_normalize_rows(const float* X, int n, int d, float eps, float* Xn, float* inv_norm, void* stream) {
  GLL_REQUIRE(X && Xn && inv_norm && n >= 1 && d >= 1 && eps > 0.f, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  GLL_PROF(KID_CONVERT, st);
  normalize_rows_kernel<<<ceil_div((long long)n * 32, 256), 256, 0, st>>>(X, n, d, eps, Xn, inv_norm);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

int gll_normalize_rows_backward(const float* Xn, const float* inv_norm, const float* dXn, int n, int d, float* dX, void* stream) {
  GLL_REQUIRE(Xn && inv_norm && dXn && dX && n >= 1 && d >= 1, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  GLL_PROF(KID_CONVERT, st);
  normalize_rows_backward_kernel<<<ceil_div((long long)n * 32, 256), 256, 0, st>>>(Xn, inv_norm, dXn, n, d, dX);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

int gll_csr_residual_f64(const int* ptr, const int* col, const double* val, const double* x, const double* b, int m, int l,
                         double* r, void* stream) {
  GLL_REQUIRE(ptr && col && val && x && b && r && m >= 1 && l >= 1, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  GLL_PROF(KID_CONVERT, st);
  csr_residual_f64_kernel<<<ceil_div((long long)m * l, 256), 256, 0, st>>>(ptr, col, val, x, b, m, l, r);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

size_t gll_cg_rows_peer_mail_bytes(void) { return cg_rows_peer_mail_bytes(); }
size_t gll_cg_rows_peer_flag_bytes(void) { return cg_rows_peer_flag_bytes(); }

int gll_cg_rows_init_p2p(const float* diag, const float* rhs, int m, int l, int row_lo, int row_hi, float* x,
                         const gll_peers* peers, unsigned epoch, void* workspace, size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(peers != nullptr, "peer table missing");
  return cg_rows_init(diag, rhs, m, l, row_lo, row_hi, x, (float*)peers->u[peers->rank], workspace, workspace_bytes, peers, epoch,
                      (cudaStream_t)stream);
}

int gll_cg_rows_spmv_p2p(const int* uu_ptr, const int* uu_col, const float* uu_val, const float* diag, int m, int l, int row_lo,
                         int row_hi, const gll_peers* peers, unsigned epoch, const int* ctrl, void* workspace,
                         size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(peers != nullptr, "peer table missing");
  return cg_rows_spmv(uu_ptr, uu_col, uu_val, diag, m, l, row_lo, row_hi, (const float*)peers->u[peers->rank], nullptr, workspace,
                      workspace_bytes, peers, epoch, ctrl, (cudaStream_t)stream);
}

int gll_cg_rows_update_p2p(const float* diag, int m, int l, int row_lo, int row_hi, int iter, int max_iter, float tol, float* x,
                           const gll_peers* peers, unsigned epoch, int* ctrl, float* resid_out, void* workspace,
                           size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(peers != nullptr, "peer table missing");
  return cg_rows_update(diag, m, l, row_lo, row_hi, nullptr, iter, max_iter, tol, x, (float*)peers->u[peers->rank], ctrl, resid_out,
                        workspace, workspace_bytes, peers, epoch, (cudaStream_t)stream);
}

int gll_ce_loss(const void* pred, int pred_is_f64, const long long* targets, int m, int l, void* loss_out, void* grad_out,
                int* status, void* workspace, size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(pred && targets && loss_out && grad_out && m >= 1 && l >= 1, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  int blocks = 1;
  if (m > 4096) {
    blocks = min(1024, min(device_info().sms * 2, ceil_div(m, 1024)));
    GLL_REQUIRE(workspace && workspace_bytes >= gll_ce_loss_workspace_bytes(m), "loss workspace too small");
  }
  double* partial = (double*)workspace;
  {
    GLL_PROF(KID_PACK, st);
    if (pred_is_f64)
      ce_loss_kernel<double><<<blocks, 1024, 0, st>>>((const double*)pred, targets, m, l, (double*)loss_out, (double*)grad_out, partial, status);
    else
      ce_loss_kernel<float><<<blocks, 1024, 0, st>>>((const float*)pred, targets, m, l, (float*)loss_out, (float*)grad_out, partial, status);
  }
  GLL_LAUNCH_CHECK();
  if (blocks > 1) {
    GLL_PROF(KID_PACK, st);
    if (pred_is_f64)
      ce_loss_finish_kernel<double><<<1, 32, 0, st>>>(partial, blocks, m, (double*)loss_out);
    else
      ce_loss_finish_kernel<float><<<1, 32, 0, st>>>(partial, blocks, m, (float*)loss_out);
    GLL_LAUNCH_CHECK();
  }
  return GLL_OK;
}

int gll_pack_columns(const float* src, int rows, int lp_src, int c0, int cnt, float* dst, int lp_dst, void* stream) {
  GLL_REQUIRE(src && dst && rows >= 1 && c0 >= 0 && cnt >= 0 && c0 + cnt <= lp_src && cnt <= lp_dst, "bad column slice");
  return pack_columns(src, rows, lp_src, c0, cnt, dst, lp_dst, (cudaStream_t)stream);
}

int gll_unpack_columns(const float* src, int rows, int lp_src, int c0, int cnt, float* dst, int lp_dst, void* stream) {
  GLL_REQUIRE(src && dst && rows >= 1 && c0 >= 0 && cnt >= 0 && cnt <= lp_src && c0 + cnt <= lp_dst, "bad column slice");
  return unpack_columns(src, rows, lp_src, c0, cnt, dst, lp_dst, (cudaStream_t)stream);
}

int gll_unpack_pred(const float* u, int m, int l, void* pred, int pred_is_f64, void* stream) {
  GLL_REQUIRE(u && pred && m >= 1 && l >= 1, "bad arguments");
  return unpack_pred(u, m, l, padded_classes(l), pred, pred_is_f64, (cudaStream_t)stream);
}

int gll_pack_grad(const void* grad_out, int grad_is_f64, int m, int l, float* rhs, void* stream) {
  GLL_REQUIRE(grad_out && rhs && m >= 1 && l >= 1, "bad arguments");
  return pack_grad(grad_out, grad_is_f64, m, l, padded_classes(l), rhs, (cudaStream_t)stream);
}

// the state's arrays and the workspace check of the fused drivers (need: the driver's workspace size)
static int driver_bufs(int n, int k, int l, int k_lab, void* state, size_t need, size_t workspace_bytes, GraphBufs* B) {
  gll_layout L;
  if (gll_state_layout(n, k, l, k_lab, &L)) return GLL_ERR_ARG;
  if (workspace_bytes < need) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, need);
    return GLL_ERR_WORKSPACE;
  }
  *B = graph_bufs(L, state);
  return GLL_OK;
}

// gll_forward after the kNN search: graph, weights and the unlabeled system from B.knn_idx / B.knn_dist, then the CG solve
static int forward_solve(const GraphBufs& B, const float* Y, int n, int k, int l, int k_lab, int eps_auto, float eps_fixed, float tau,
                         float cg_tol, int cg_max_iter, void* pred_out, int pred_is_f64, void* workspace, size_t workspace_bytes,
                         cudaStream_t st) {
  const int m = n - k_lab, lp = padded_classes(l);
  int rc = graph_stages_run(B, Y, n, k, l, k_lab, eps_auto, eps_fixed, tau, 0, 6, workspace, workspace_bytes, st);
  if (rc) return rc;
  CgSolve S = cg_system(B, m, l, cg_tol, cg_max_iter);
  S.x = B.ut + (size_t)k_lab * lp;
  S.iters_out = B.info + GLL_INFO_CG_ITERS_FWD;
  S.resid_out = (float*)(B.info + GLL_INFO_CG_RESID_FWD);
  S.status_out = B.info + GLL_INFO_STATUS;
  S.x_copy = pred_out;  // Pred (GLL.py:66) is written by the solver itself
  S.x_copy_f64 = pred_is_f64;
  S.uu_degree_hint = uu_degree_hint(n, k, m);
  return cg_run(S, workspace, workspace_bytes, st);
}

int gll_forward(const float* X, const float* Y, int n, int d, int k, int l, int k_lab, int eps_auto, float eps_fixed,
                float tau, float cg_tol, int cg_max_iter, void* state, void* pred_out, int pred_is_f64, void* workspace,
                size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(X && state && pred_out && workspace, "null pointer");
  GraphBufs B;
  int rc = driver_bufs(n, k, l, k_lab, state, gll_workspace_bytes(n, d, k, l, k_lab), workspace_bytes, &B);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  GLL_CUDA_CHECK(cudaMemsetAsync(B.info, 0, sizeof(int) * GLL_INFO_WORDS, st));
  rc = knn_run(X, n, d, k, 0, n, B.knn_idx, B.knn_dist, B.info, workspace, workspace_bytes, st);
  if (rc) return rc;
  return forward_solve(B, Y, n, k, l, k_lab, eps_auto, eps_fixed, tau, cg_tol, cg_max_iter, pred_out, pred_is_f64, workspace,
                       workspace_bytes, st);
}

size_t gll_knn_segments_workspace_bytes(int n, int d, int k, const int* seg_ptr_host, int nseg) {
  return knn_seg_ws_bytes(n, d, k, seg_ptr_host, nseg);
}

int gll_knn_segments(const float* X, int n, int d, int k, const int* seg_ptr_host, int nseg, int* knn_idx, float* knn_dist, int* info,
                     void* workspace, size_t workspace_bytes, void* stream) {
  return knn_run_segments(X, n, d, k, seg_ptr_host, nseg, knn_idx, knn_dist, info, workspace, workspace_bytes, (cudaStream_t)stream);
}

void gll_knn_segments_units(int n, int d, const int* seg_ptr_host, int nseg, long long* seg_units, long long* uniform_units) {
  long long a = 0, b = 0;
  knn_seg_units(n, d, seg_ptr_host, nseg, &a, &b);
  if (seg_units) *seg_units = a;
  if (uniform_units) *uniform_units = b;
}

// k <= 33: the segmented search serves one candidate round (gll_knn_segments)
static bool batched_sizes_ok(int B, int n, int d, int k, int l, int k_lab) {
  return B >= 1 && n >= k && k >= 2 && k <= 33 && d >= 1 && l >= 1 && k_lab >= 1 && k_lab < n && (long long)B * n <= 0x7fffffffLL;
}

static std::vector<int> uniform_segments(int B, int n) {
  std::vector<int> seg(B + 1);
  for (int b = 0; b <= B; ++b) seg[b] = b * n;
  return seg;
}

}  // extern "C"

namespace gll {

// the segmented search's lists in natural order, in front of the search's own workspace; returns their bytes (ws == NULL: size
// query only)
static size_t batched_lists(void* ws, int N, int k, int** idx, float** dist) {
  Carver cv(ws, ~(size_t)0);
  int* i = cv.take<int>((size_t)N * k);
  float* x = cv.take<float>((size_t)N * k);
  if (idx) *idx = i;
  if (dist) *dist = x;
  return align_up(cv.off, 256);
}

size_t batched_ws_bytes(int B, int n, int d, int k, int l, int k_lab) {
  const int N = B * n;
  const std::vector<int> seg = uniform_segments(B, n);
  const size_t s = knn_seg_ws_bytes(N, d, k, seg.data(), B);
  if (s == 0) return 0;
  size_t b = batched_lists(nullptr, N, k, nullptr, nullptr) + s;
  b = std::max(b, graph_weights_ws_bytes(N, k));
  return std::max(b, cg_ws_bytes(N - B * k_lab, l));
}

int batched_knn_run(const float* X, int B, int n, int d, int k, int k_lab, const GraphBufs& G, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int N = B * n;
  int* idx;
  float* dist;
  const size_t lists = batched_lists(ws, N, k, &idx, &dist);
  const std::vector<int> seg = uniform_segments(B, n);
  const int rc = knn_run_segments(X, N, d, k, seg.data(), B, idx, dist, G.info, (char*)ws + lists, ws_bytes - lists, st);
  if (rc) return rc;
  {
    GLL_PROF(KID_BATCH_REORDER, st);
    knn_to_labeled_first_kernel<<<ceil_div((long long)N * k, 256), 256, 0, st>>>(idx, dist, B, n, k, k_lab, G.knn_idx, G.knn_dist);
  }
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

}  // namespace gll

extern "C" {

size_t gll_batched_workspace_bytes(int B, int n, int d, int k, int l, int k_lab) {
  if (!batched_sizes_ok(B, n, d, k, l, k_lab)) return 0;
  return batched_ws_bytes(B, n, d, k, l, k_lab);
}

int gll_forward_batched(const float* X, const float* Y, int B, int n, int d, int k, int l, int k_lab, int eps_auto, float eps_fixed,
                        float tau, float cg_tol, int cg_max_iter, void* state, void* pred_out, int pred_is_f64, void* workspace,
                        size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(X && Y && state && pred_out && workspace, "null pointer");
  GLL_REQUIRE(batched_sizes_ok(B, n, d, k, l, k_lab), "need B >= 1, 2 <= k <= 33, n >= k, 1 <= k_lab < n, B n < 2^31");
  const int N = B * n, K = B * k_lab;
  GraphBufs G;
  int rc = driver_bufs(N, k, l, K, state, gll_batched_workspace_bytes(B, n, d, k, l, k_lab), workspace_bytes, &G);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  GLL_CUDA_CHECK(cudaMemsetAsync(G.info, 0, sizeof(int) * GLL_INFO_WORDS, st));
  rc = batched_knn_run(X, B, n, d, k, k_lab, G, workspace, workspace_bytes, st);
  if (rc) return rc;
  return forward_solve(G, Y, N, k, l, K, eps_auto, eps_fixed, tau, cg_tol, cg_max_iter, pred_out, pred_is_f64, workspace, workspace_bytes,
                       st);
}

int gll_backward(const float* X, const void* grad_out, int grad_is_f64, int n, int d, int k, int l, int k_lab, int eps_auto,
                 float cg_tol, int cg_max_iter, void* state, float* dX, void* workspace, size_t workspace_bytes,
                 void* stream) {
  return gll_backward_scaled(X, grad_out, grad_is_f64, nullptr, 0, n, d, k, l, k_lab, eps_auto, cg_tol, cg_max_iter, state, dX, workspace,
                             workspace_bytes, stream);
}

int gll_backward_scaled(const float* X, const void* grad_out, int grad_is_f64, const void* scale, int scale_is_f64, int n, int d, int k,
                        int l, int k_lab, int eps_auto, float cg_tol, int cg_max_iter, void* state, float* dX, void* workspace,
                        size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(X && grad_out && state && dX && workspace, "null pointer");
  GraphBufs B;
  int rc = driver_bufs(n, k, l, k_lab, state, gll_workspace_bytes(n, d, k, l, k_lab), workspace_bytes, &B);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int m = n - k_lab, lp = padded_classes(l);
  // GLL.py:104: the solver reads the incoming gradient itself; the labeled rows of the padded adjoint solution (zeros) are
  // never read -- edge_grad substitutes them
  CgSolve S = cg_system(B, m, l, cg_tol, cg_max_iter);
  S.x = B.wt + (size_t)k_lab * lp;
  S.iters_out = B.info + GLL_INFO_CG_ITERS_BWD;
  S.resid_out = (float*)(B.info + GLL_INFO_CG_RESID_BWD);
  S.status_out = B.info + GLL_INFO_STATUS;
  S.rhs_src = grad_out;
  S.rhs_kind = grad_is_f64 ? 2 : 1;
  S.rhs_scale = scale;
  S.rhs_scale_f64 = scale_is_f64;
  S.uu_degree_hint = uu_degree_hint(n, k, m);
  rc = cg_run(S, workspace, workspace_bytes, st);
  if (rc) return rc;
  return backward_edges_run(X, n, d, l, k_lab, eps_auto, B, dX, 0, n, 3, st);
}

}  // extern "C"
