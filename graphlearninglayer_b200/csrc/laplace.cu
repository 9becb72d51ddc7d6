// Laplace-learning evaluation on the device (utils.py:570-593 `laplace`, used by test_GL_NP at utils.py:637-660):
// features -> graph -> harmonic extension refined in fp64 to the reference's stop rule -> argmax labels and a hit count.
//
//   gll_laplace_eval:  K1 + K2/K3 (gll_forward's stages with the caller's k)
//                      fp32 Jacobi-CG  (L_uu + tau I) x0 = -L_ul Y,  relative tolerance GLL_LAPLACE_CG_RTOL0
//                      GLL_LAPLACE_ROUNDS x { laplace_refine ; fp32 correction CG at GLL_LAPLACE_CG_RTOL }
//                      laplace_finish
//
// laplace_refine (round r) reads x_{r-1} (fp64) and the previous fp32 correction e_{r-1}, and writes x_r = x_{r-1} + e_{r-1}
// to the OTHER fp64 buffer (neighbour rows are read while rows are written, so the rounds ping-pong between `pred` and a
// workspace buffer).  In the same pass it forms the fp64 residual over the full-graph CSR,
//     r_i = sum_j w_ij (u_j - x_i) - tau x_i,   u = [Y; x_r],
// i.e. b - A x with A = D - W_uu + tau I, D = ROW sums of the stored fp32 weights accumulated in fp64, and the reference's
// stop quantity per class column ||M r_c||_2 = sqrt(sum_i r_ic^2 / (D_i + tau + 1e-10)) (make_golden_eval.py:41-45).
// Per-CTA column partials are added in CTA order by the last CTA (integer ticket): no floating-point atomics.  That CTA
// writes the correction solve's right-hand-side scale: 1 while some column is above tol, else 0 -- a zero right-hand side
// stops every CG kernel at iteration 0 and the correction is exactly zero, so the round count is fixed and no host decision
// is needed.  laplace_finish adds the last correction, writes pred, the argmax labels and the hit count.
#include <algorithm>

#include "cg_common.cuh"
#include "common.cuh"

namespace gll {
namespace {

constexpr int LR_THREADS = 256;

struct RefineParams {
  const int* row_ptr;  // full graph, n rows
  const int* col;
  const float* w;
  const float* Y;        // k_lab x l
  const double* x_prev;  // m x l, or NULL (round 0)
  const float* e;        // m x lp fp32 correction (round 0: the initial solution)
  double* x_out;         // m x l
  double* r_out;         // m x l: right-hand side of the correction solve
  double* partial;       // [B][gx][l]
  double* colnorm;       // [B][l]
  double* gmax;          // [B]: per graph, the largest column norm (NaN: a column is not finite)
  double* resid;         // [B] or NULL: the caller's copy of gmax
  double* scale;         // 1 scalar
  unsigned* ticket;      // [B + 1]: CTAs done per graph, then graphs done
  int* info;
  int n, k_lab, m, mb, B, gx, l, lp, cw, round;
  double tau, tol;
};

// B graphs whose unlabeled rows are the consecutive ranges [b mb, (b + 1) mb) of the m = B mb unlabeled rows (B = 1: one graph).
// Block = RL row lanes x CW class columns (CW = min(l, 32)); blockIdx.x = b gx + (CTA of graph b), blockIdx.y picks a chunk of CW
// columns.  A thread walks the rows of its lane in graph b in a fixed order and keeps its own partial sum of r^2 / diag: the
// reduction order depends on nothing but the launch shape.  The last CTA of graph b (integer ticket) adds that graph's per-CTA
// column partials in CTA order and writes the graph's largest column norm; the last graph to finish takes the maximum over
// graphs, which decides the correction scale and the info slots.  No floating-point atomics.
__global__ void __launch_bounds__(LR_THREADS) laplace_refine_kernel(RefineParams P) {
  __shared__ double red[LR_THREADS];
  __shared__ bool last;
  const int cw = P.cw, rl_count = LR_THREADS / cw;
  const int tid = threadIdx.x, rl = tid / cw, cc = tid - rl * cw;
  const int c = blockIdx.y * cw + cc;
  const int b = blockIdx.x / P.gx, bx = blockIdx.x - b * P.gx;
  const bool active = rl < rl_count && c < P.l;
  double acc = 0.0;
  if (active) {
    const int l = P.l, lp = P.lp, k_lab = P.k_lab, i_end = (b + 1) * P.mb;
    for (int i = b * P.mb + bx * rl_count + rl; i < i_end; i += P.gx * rl_count) {
      const size_t o = (size_t)i * l + c;
      const double xi = (P.x_prev ? __ldg(P.x_prev + o) : 0.0) + (double)__ldg(P.e + (size_t)i * lp + c);
      P.x_out[o] = xi;
      const int g = k_lab + i, e1 = __ldg(P.row_ptr + g + 1);
      double s = 0.0, deg = 0.0;
      for (int e = __ldg(P.row_ptr + g); e < e1; ++e) {
        const int j = __ldg(P.col + e);
        const double wv = (double)__ldg(P.w + e);
        double uj;
        if (j < k_lab) {
          uj = (double)__ldg(P.Y + (size_t)j * l + c);
        } else {
          const int jj = j - k_lab;
          uj = (P.x_prev ? __ldg(P.x_prev + (size_t)jj * l + c) : 0.0) + (double)__ldg(P.e + (size_t)jj * lp + c);
        }
        s = fma(wv, uj - xi, s);
        deg += wv;
      }
      const double r = s - P.tau * xi;
      P.r_out[o] = r;
      acc = fma(r, r / (deg + P.tau + 1e-10), acc);
    }
  }
  red[tid] = acc;
  __syncthreads();
  if (tid < cw && c < P.l) {
    double t = 0.0;
    for (int q = 0; q < rl_count; ++q) t += red[q * cw + tid];
    P.partial[(size_t)blockIdx.x * P.l + c] = t;
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) last = atomicAdd(P.ticket + b, 1u) == P.gx * gridDim.y - 1u;
  __syncthreads();
  if (!last) return;
  __threadfence();
  const int lane = tid & 31, warp = tid >> 5;
  const double* part = P.partial + (size_t)b * P.gx * P.l;
  double* colnorm = P.colnorm + (size_t)b * P.l;
  for (int cc2 = warp; cc2 < P.l; cc2 += LR_THREADS / 32) {
    double t = 0.0;
    for (int q = lane; q < P.gx; q += 32) t += __ldcg(part + (size_t)q * P.l + cc2);
    t = warp_sum(t);
    if (lane == 0) colnorm[cc2] = sqrt(t);
  }
  __syncthreads();
  if (tid == 0) {
    double mx = 0.0;
    bool bad = false;
    for (int cc2 = 0; cc2 < P.l; ++cc2) {
      const double v = colnorm[cc2];
      if (!(v == v) || isinf(v)) bad = true;
      mx = fmax(mx, v);
    }
    const double gv = bad ? __longlong_as_double(0x7ff8000000000000LL) : mx;
    P.gmax[b] = gv;
    if (P.resid != nullptr) P.resid[b] = gv;
    P.ticket[b] = 0u;  // rewound for the next round
    __threadfence();
    last = atomicAdd(P.ticket + P.B, 1u) == (unsigned)P.B - 1u;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  // maximum over graphs: exact, so the order of the reduction does not matter
  double mx = 0.0;
  bool bad = false;
  for (int g = tid; g < P.B; g += LR_THREADS) {
    const double v = __ldcg(P.gmax + g);
    if (!(v == v)) bad = true;
    mx = fmax(mx, v);
  }
  bad = __syncthreads_or(bad) != 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(FULL, mx, o));
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < LR_THREADS / 32; ++w) mx = fmax(mx, red[w]);
    const bool more = bad || !(mx <= P.tol);
    *P.scale = more ? 1.0 : 0.0;
    if (more) P.info[GLL_INFO_LAPLACE_ROUNDS] = P.round + 1;
    if (bad) atomicOr(P.info + GLL_INFO_STATUS, GLL_STATUS_NONFINITE);
    const float fr = bad ? __int_as_float(0x7fc00000) : (float)mx;
    P.info[GLL_INFO_LAPLACE_RESID] = __float_as_int(fr);
    if (P.round == 0) P.info[GLL_INFO_LAPLACE_RESID0] = __float_as_int(fr);
    P.ticket[P.B] = 0u;
  }
}

// Thread per unlabeled row: pred = x + e (in place), labels = first maximal column, hits counted with one integer atomic per CTA
// into correct[b].  The fb CTAs of graph b cover its rows [b mb, (b + 1) mb).  CTA 0 also writes the correction-CG iteration
// counts and the convergence status.
__global__ void __launch_bounds__(LR_THREADS)
laplace_finish_kernel(double* __restrict__ pred, const float* __restrict__ e, int mb, int fb, int l, int lp, long long* __restrict__ labels,
                      const long long* __restrict__ targets, unsigned long long* __restrict__ correct, const double* __restrict__ scale,
                      const int* __restrict__ round_iters, int rounds, int* __restrict__ info) {
  __shared__ int part[LR_THREADS / 32];
  const int b = blockIdx.x / fb, t = (blockIdx.x - b * fb) * blockDim.x + threadIdx.x, i = b * mb + t;
  int hit = 0;
  if (t < mb) {
    double best = 0.0;
    int arg = 0;
    for (int c = 0; c < l; ++c) {
      const size_t o = (size_t)i * l + c;
      const double v = pred[o] + (double)__ldg(e + (size_t)i * lp + c);
      pred[o] = v;
      if (c == 0 || v > best) {
        best = v;
        arg = c;
      }
    }
    labels[i] = arg;
    if (targets != nullptr) {
      const long long tg = __ldg(targets + i);
      hit = (tg >= 0 && tg == (long long)arg) ? 1 : 0;
    }
  }
  if (correct != nullptr) {
    hit = warp_sum(hit);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = hit;
    __syncthreads();
    if (threadIdx.x == 0) {
      int s = 0;
      for (int w = 0; w < LR_THREADS / 32; ++w) s += part[w];
      if (s) atomicAdd(correct + b, (unsigned long long)s);
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    int tot = 0;
    unsigned packed[2] = {0u, 0u};
    for (int r = 0; r < rounds; ++r) {
      const int it = round_iters[r];
      tot += it;
      if (r < 4) packed[r >> 1] |= (unsigned)min(it, 65535) << (16 * (r & 1));
    }
    info[GLL_INFO_LAPLACE_CG_ITERS] = tot;
    info[GLL_INFO_LAPLACE_ROUND_ITERS] = (int)packed[0];
    info[GLL_INFO_LAPLACE_ROUND_ITERS + 1] = (int)packed[1];
    if (*scale != 0.0) atomicOr(info + GLL_INFO_STATUS, GLL_STATUS_CG_NOT_CONVERGED);  // tol unmet after the last round
  }
}

// CTAs per graph of laplace_refine (mb unlabeled rows per graph)
int refine_grid_x(int mb, int l) {
  const int cw = min(l, 32), rl = LR_THREADS / cw;
  return max(1, min(ceil_div(mb, rl), 4 * device_info().sms));
}

// the evaluation's own buffers, behind the layer state and in front of the stage workspace
struct EvalBufs {
  double* xtmp;    // m x l
  double* r;       // m x l
  double* partial; // [B][refine grid][l]
  double* colnorm; // [B][l]
  double* gmax;    // [B]
  double* scale;
  unsigned* ticket;  // [B + 1]
  int* round_iters;  // [GLL_LAPLACE_ROUNDS]
};

// base == NULL: size query only
size_t eval_bufs(char* base, int B, int mb, int l, EvalBufs* E) {
  Carver cv(base, ~(size_t)0);
  const size_t m = (size_t)B * mb;
  EvalBufs b;
  b.xtmp = cv.take<double>(m * l);
  b.r = cv.take<double>(m * l);
  b.partial = cv.take<double>((size_t)B * refine_grid_x(mb, l) * l);
  b.colnorm = cv.take<double>((size_t)B * l);
  b.gmax = cv.take<double>(B);
  b.scale = cv.take<double>(1);
  b.ticket = cv.take<unsigned>((size_t)B + 1);
  b.round_iters = cv.take<int>(GLL_LAPLACE_ROUNDS);
  if (E) *E = b;
  return align_up(cv.off, 256);
}

// workspace of B graphs of n rows: [layer state of the union | the evaluation's buffers | stage workspace]; 0 for sizes the stages
// refuse
size_t eval_ws_bytes(int B, int n, int d, int k, int l, int k_lab) {
  gll_layout L;
  if (gll_state_layout(B * n, k, l, B * k_lab, &L)) return 0;
  const size_t stage = (B == 1) ? gll_workspace_bytes(n, d, k, l, k_lab) : batched_ws_bytes(B, n, d, k, l, k_lab);
  if (stage == 0) return 0;
  return L.total + eval_bufs(nullptr, B, n - k_lab, l, nullptr) + stage;
}

// the sizes gll_laplace_eval_batched accepts
bool eval_batched_sizes_ok(int B, int n, int d, int k, int l, int k_lab) {
  if (B < 1 || n < 1 || (long long)B * n > 0x7fffffffLL) return false;
  return k >= 2 && k <= 64 && k <= n && (k <= 33 || (long long)B * n >= 256) && d >= 1 && l >= 1 && k_lab >= 1 && k_lab < n;
}

// gll_laplace_eval (B = 1) and gll_laplace_eval_batched: sizes are checked by the callers
int eval_run(const float* X, const float* Y, int B, int n, int d, int k, int l, int k_lab, int eps_auto, float eps_fixed, float tau,
             double tol, int cg_max_iter, double* pred, long long* labels, const long long* targets, long long* correct_out,
             double* resid_out, int* info, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const size_t need = eval_ws_bytes(B, n, d, k, l, k_lab);
  if (workspace_bytes < need) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, need);
    return GLL_ERR_WORKSPACE;
  }
  const int N = B * n, K = B * k_lab, mb = n - k_lab, m = N - K, lp = padded_classes(l);
  gll_layout L;
  if (gll_state_layout(N, k, l, K, &L)) return GLL_ERR_ARG;
  // workspace = [layer state | the evaluation's buffers | stage workspace]
  char* S = (char*)workspace;
  GraphBufs G = graph_bufs(L, S);
  G.info = info;  // the caller's info block in place of the state's
  EvalBufs E;
  const size_t eb = eval_bufs(S + L.total, B, mb, l, &E);
  void* ws = S + L.total + eb;
  const size_t ws_bytes = workspace_bytes - L.total - eb;

  GLL_CUDA_CHECK(cudaMemsetAsync(info, 0, sizeof(int) * GLL_INFO_WORDS, st));
  GLL_CUDA_CHECK(cudaMemsetAsync(E.ticket, 0, sizeof(unsigned) * ((size_t)B + 1), st));
  if (correct_out) GLL_CUDA_CHECK(cudaMemsetAsync(correct_out, 0, sizeof(long long) * (size_t)B, st));
  int rc = (B == 1) ? knn_run(X, n, d, k, 0, n, G.knn_idx, G.knn_dist, info, ws, ws_bytes, st)
                    : batched_knn_run(X, B, n, d, k, k_lab, G, ws, ws_bytes, st);
  if (rc) return rc;
  rc = graph_stages_run(G, Y, N, k, l, K, eps_auto, eps_fixed, tau, 0, 6, ws, ws_bytes, st);
  if (rc) return rc;
  float* x0 = G.ut + (size_t)K * lp;
  float* corr = G.wt;  // the adjoint's region, free in an evaluation
  unsigned* barrier = (unsigned*)(info + GLL_INFO_CG_BARRIER);  // zeroed with info, rewound by the kernels
  // No sparsity hint (0): the evaluation system is never routed to the cluster kernel.  No status pointer either: an inner solve
  // that stops at the fp32 floor is not a failure -- the fp64 rounds decide convergence.  B graphs are one block-diagonal system:
  // every CG solves them together, with step lengths shared by the graphs (per class column).
  rc = cg_run(G.uu_ptr, G.uu_col, G.uu_val, G.diag, G.rhs, m, l, -(float)GLL_LAPLACE_CG_RTOL0, cg_max_iter, x0,
              info + GLL_INFO_CG_ITERS_FWD, (float*)(info + GLL_INFO_CG_RESID_FWD), nullptr, ws, ws_bytes, st, barrier, nullptr);
  if (rc) return rc;

  RefineParams P;
  P.row_ptr = G.row_ptr;
  P.col = G.col;
  P.w = G.w;
  P.Y = Y;
  P.r_out = E.r;
  P.partial = E.partial;
  P.colnorm = E.colnorm;
  P.gmax = E.gmax;
  P.resid = resid_out;
  P.scale = E.scale;
  P.ticket = E.ticket;
  P.info = info;
  P.n = N;
  P.k_lab = K;
  P.m = m;
  P.mb = mb;
  P.B = B;
  P.gx = refine_grid_x(mb, l);
  P.l = l;
  P.lp = lp;
  P.cw = min(l, 32);
  P.tau = (double)tau;
  P.tol = tol;
  const dim3 grid(B * P.gx, ceil_div(l, P.cw));
  const CgIo io = {E.r, 2, nullptr, 0, E.scale, 1, 0.f};
  for (int r = 0; r < GLL_LAPLACE_ROUNDS; ++r) {
    // the last round writes pred; rounds alternate between pred and the workspace buffer
    double* out = ((GLL_LAPLACE_ROUNDS - 1 - r) % 2 == 0) ? pred : E.xtmp;
    P.x_prev = (r == 0) ? nullptr : (out == pred ? E.xtmp : pred);
    P.e = (r == 0) ? x0 : corr;
    P.x_out = out;
    P.round = r;
    {
      GLL_PROF(KID_LAPLACE_REFINE, st);
      laplace_refine_kernel<<<grid, LR_THREADS, 0, st>>>(P);
      GLL_LAUNCH_CHECK();
    }
    rc = cg_run(G.uu_ptr, G.uu_col, G.uu_val, G.diag, G.rhs, m, l, -(float)GLL_LAPLACE_CG_RTOL, cg_max_iter, corr, E.round_iters + r,
                nullptr, nullptr, ws, ws_bytes, st, barrier, &io);
    if (rc) return rc;
  }
  {
    GLL_PROF(KID_LAPLACE_FINISH, st);
    const int fb = ceil_div(mb, LR_THREADS);
    laplace_finish_kernel<<<B * fb, LR_THREADS, 0, st>>>(pred, corr, mb, fb, l, lp, labels, targets, (unsigned long long*)correct_out,
                                                         E.scale, E.round_iters, GLL_LAPLACE_ROUNDS, info);
    GLL_LAUNCH_CHECK();
  }
  return GLL_OK;
}

// ---------------------------------------------------------------------------------------------- T trials on one graph
// gll_laplace_eval_trials: trial t clamps the k_lab rows train_idx[t] to the label rows Y[t] and solves the other rows.  The graph
// is the same in every trial, so the stages run once with k_lab = 0: the system is the FULL graph A = D + tau I - W over all n
// rows, and trial t masks its clamped rows out of its own columns (cg_persistent_kernel<true>: A p is zeroed there, so r, p and
// x stay 0 on those rows).  Every [n][C] array has C = T lpad columns, lpad = padded_classes(l): trial t owns the columns
// [t lpad, t lpad + l), so a class quad never spans two trials.  slot[i T + t] = s when train_idx[t, s] == i, else -1.

// slot / bad from train_idx: slot is -1 on entry (memset), bad zero.  An index outside [0, n) or a repeat (the atomicCAS from -1
// fails) makes the trial invalid; no index is used before it has been checked.
__global__ void laplace_trials_setup_kernel(const void* __restrict__ idx, int is_i64, int n, int T, int k_lab, int* __restrict__ slot,
                                            int* __restrict__ bad, int* __restrict__ info) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= (long long)T * k_lab) return;
  const int t = (int)(q / k_lab), s = (int)(q - (long long)t * k_lab);
  const long long i = is_i64 ? __ldg(reinterpret_cast<const long long*>(idx) + q) : (long long)__ldg(reinterpret_cast<const int*>(idx) + q);
  bool ok = i >= 0 && i < n;
  if (ok) ok = atomicCAS(slot + (size_t)i * T + t, -1, s) == -1;
  if (!ok) {
    bad[t] = 1;
    atomicOr(info + GLL_INFO_STATUS, GLL_STATUS_BAD_INDEX);
  }
}

struct TrialsRefineParams {
  const int* row_ptr;  // full graph, n rows
  const int* col;
  const float* w;
  const float* Y;        // T x k_lab x l
  const int* slot;       // [n][T]
  const int* bad;        // [T]
  const double* x_prev;  // [n][C], or NULL
  const float* e;        // [n][C] fp32 correction (round 0: the initial solution), or NULL: x = 0
  double* x_out;         // [n][C], or NULL
  double* r_out;         // [n][C]: right-hand side of the next solve (padding columns stay 0)
  double* partial;       // [gx][T l]
  double* colnorm;       // [T l]
  double* resid;         // [T] or NULL
  double* scale;         // 1 scalar
  unsigned* ticket;      // 1
  int* info;
  int n, T, k_lab, l, lpad, gx, cw, round;  // round < 0: r = b only (x = 0), no stop-rule bookkeeping
  double tau, tol;
};

// laplace_refine_kernel per (row, trial column): block = RL row lanes x CW of the T l class columns, blockIdx.y picks the chunk of
// CW columns.  A row clamped in trial t, and every row of an invalid trial, has r = 0; a neighbour j clamped in trial t reads
// u_j = Y[t, slot], the others the iterate.  Column partials are added in CTA order by the last CTA (one integer ticket); it
// writes each valid trial's largest column norm (resid: NaN for an invalid trial), and the correction scale is 1 while any
// column of any valid trial is above tol.  No floating-point atomics.
__global__ void __launch_bounds__(LR_THREADS) laplace_refine_trials_kernel(TrialsRefineParams P) {
  __shared__ double red[LR_THREADS];
  __shared__ bool last;
  const int cw = P.cw, rl_count = LR_THREADS / cw, TL = P.T * P.l;
  const int tid = threadIdx.x, rl = tid / cw, cc = tid - rl * cw;
  const int c = blockIdx.y * cw + cc;
  const bool active = rl < rl_count && c < TL;
  double acc = 0.0;
  if (active) {
    const int T = P.T, l = P.l, t = c / l, cl = c - t * l;
    const size_t C = (size_t)T * P.lpad, sc = (size_t)t * P.lpad + cl;
    const float* Yt = P.Y + (size_t)t * P.k_lab * l + cl;
    const bool valid = __ldg(P.bad + t) == 0;
    for (int i = blockIdx.x * rl_count + rl; i < P.n; i += P.gx * rl_count) {
      const size_t o = (size_t)i * C + sc;
      const double xi = (P.x_prev ? __ldg(P.x_prev + o) : 0.0) + (P.e ? (double)__ldg(P.e + o) : 0.0);
      if (P.x_out) P.x_out[o] = xi;
      if (!valid || __ldg(P.slot + (size_t)i * T + t) >= 0) {
        P.r_out[o] = 0.0;
        continue;
      }
      const int e1 = __ldg(P.row_ptr + i + 1);
      double s = 0.0, deg = 0.0;
      for (int e = __ldg(P.row_ptr + i); e < e1; ++e) {
        const int j = __ldg(P.col + e);
        const double wv = (double)__ldg(P.w + e);
        const int sj = __ldg(P.slot + (size_t)j * T + t);
        const size_t oj = (size_t)j * C + sc;
        const double uj = (sj >= 0) ? (double)__ldg(Yt + (size_t)sj * l)
                                    : (P.x_prev ? __ldg(P.x_prev + oj) : 0.0) + (P.e ? (double)__ldg(P.e + oj) : 0.0);
        s = fma(wv, uj - xi, s);
        deg += wv;
      }
      const double r = s - P.tau * xi;
      P.r_out[o] = r;
      acc = fma(r, r / (deg + P.tau + 1e-10), acc);
    }
  }
  if (P.round < 0) return;  // grid-uniform
  red[tid] = acc;
  __syncthreads();
  if (tid < cw && c < TL) {
    double t = 0.0;
    for (int q = 0; q < rl_count; ++q) t += red[q * cw + tid];
    P.partial[(size_t)blockIdx.x * TL + c] = t;
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) last = atomicAdd(P.ticket, 1u) == P.gx * gridDim.y - 1u;
  __syncthreads();
  if (!last) return;
  __threadfence();
  const int lane = tid & 31, warp = tid >> 5;
  for (int c2 = warp; c2 < TL; c2 += LR_THREADS / 32) {
    double t = 0.0;
    for (int q = lane; q < P.gx; q += 32) t += __ldcg(P.partial + (size_t)q * TL + c2);
    t = warp_sum(t);
    if (lane == 0) P.colnorm[c2] = sqrt(t);
  }
  __syncthreads();
  // per trial the largest column norm; the maximum over valid trials is exact, so its order does not matter
  double mx = 0.0;
  bool bad = false;
  for (int t = tid; t < P.T; t += LR_THREADS) {
    double tm = 0.0;
    bool tb = false;
    for (int c2 = t * P.l; c2 < (t + 1) * P.l; ++c2) {
      const double v = P.colnorm[c2];
      if (!(v == v) || isinf(v)) tb = true;
      tm = fmax(tm, v);
    }
    const bool valid = __ldg(P.bad + t) == 0;
    if (P.resid != nullptr) P.resid[t] = (tb || !valid) ? __longlong_as_double(0x7ff8000000000000LL) : tm;
    if (valid) {
      bad = bad || tb;
      mx = fmax(mx, tm);
    }
  }
  bad = __syncthreads_or(bad) != 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(FULL, mx, o));
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < LR_THREADS / 32; ++w) mx = fmax(mx, red[w]);
    const bool more = bad || !(mx <= P.tol);
    *P.scale = more ? 1.0 : 0.0;
    if (more) P.info[GLL_INFO_LAPLACE_ROUNDS] = P.round + 1;
    if (bad) atomicOr(P.info + GLL_INFO_STATUS, GLL_STATUS_NONFINITE);
    const float fr = bad ? __int_as_float(0x7fc00000) : (float)mx;
    P.info[GLL_INFO_LAPLACE_RESID] = __float_as_int(fr);
    if (P.round == 0) P.info[GLL_INFO_LAPLACE_RESID0] = __float_as_int(fr);
    *P.ticket = 0u;  // rewound for the next round
  }
}

// Thread per (row i, trial t = blockIdx.y): pred[t, i] = x + e, or the label row where i is clamped in t, or NaN for an invalid
// trial; labels = first maximal column (-1 for an invalid trial); hits of the unclamped rows counted with one integer atomic per
// CTA into correct[t] (-1 for an invalid trial).  CTA (0, 0) also writes the correction-CG iteration counts and the status.
__global__ void __launch_bounds__(LR_THREADS)
laplace_finish_trials_kernel(const double* __restrict__ x, const float* __restrict__ e, const float* __restrict__ Y,
                             const int* __restrict__ slot, const int* __restrict__ badv, int n, int T, int k_lab, int l, int lpad,
                             double* __restrict__ pred, long long* __restrict__ labels, const long long* __restrict__ targets,
                             unsigned long long* __restrict__ correct, const double* __restrict__ scale,
                             const int* __restrict__ round_iters, int rounds, int* __restrict__ info) {
  __shared__ int part[LR_THREADS / 32];
  const int t = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = __ldg(badv + t) == 0;
  int hit = 0;
  if (i < n) {
    double* p = pred + ((size_t)t * n + i) * l;
    long long arg = -1;
    if (!valid) {
      for (int c = 0; c < l; ++c) p[c] = __longlong_as_double(0x7ff8000000000000LL);
    } else {
      const int si = __ldg(slot + (size_t)i * T + t);
      const size_t o = (size_t)i * T * lpad + (size_t)t * lpad;
      const float* y = Y + ((size_t)t * k_lab + (si >= 0 ? si : 0)) * l;
      double best = 0.0;
      for (int c = 0; c < l; ++c) {
        const double v = (si >= 0) ? (double)__ldg(y + c) : x[o + c] + (double)__ldg(e + o + c);
        p[c] = v;
        if (c == 0 || v > best) {
          best = v;
          arg = c;
        }
      }
      if (si < 0 && targets != nullptr) {
        const long long tg = __ldg(targets + i);
        hit = (tg >= 0 && tg == arg) ? 1 : 0;
      }
    }
    labels[(size_t)t * n + i] = arg;
  }
  if (correct != nullptr) {
    hit = warp_sum(hit);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = hit;
    __syncthreads();
    if (threadIdx.x == 0) {
      int s = 0;
      for (int w = 0; w < LR_THREADS / 32; ++w) s += part[w];
      if (!valid) {
        if (blockIdx.x == 0) correct[t] = ~0ull;  // -1; no other CTA of an invalid trial adds anything
      } else if (s) {
        atomicAdd(correct + t, (unsigned long long)s);
      }
    }
  }
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
    int tot = 0;
    unsigned packed[2] = {0u, 0u};
    for (int r = 0; r < rounds; ++r) {
      const int it = round_iters[r];
      tot += it;
      if (r < 4) packed[r >> 1] |= (unsigned)min(it, 65535) << (16 * (r & 1));
    }
    info[GLL_INFO_LAPLACE_CG_ITERS] = tot;
    info[GLL_INFO_LAPLACE_ROUND_ITERS] = (int)packed[0];
    info[GLL_INFO_LAPLACE_ROUND_ITERS + 1] = (int)packed[1];
    if (*scale != 0.0) atomicOr(info + GLL_INFO_STATUS, GLL_STATUS_CG_NOT_CONVERGED);  // tol unmet after the last round
  }
}

// launch shape of laplace_refine_trials_kernel: CW columns per CTA, column chunks, and row CTAs (about 4 CTAs per SM in all, so
// the last CTA adds few partials per column)
struct TrialsGrid {
  int cw, gy, gx;
};
TrialsGrid trials_grid(int n, int T, int l) {
  const int tl = T * l, cw = min(tl, 32), gy = ceil_div(tl, cw);
  return {cw, gy, max(1, min(ceil_div(n, LR_THREADS / cw), ceil_div(4 * device_info().sms, gy)))};
}

// the trials' own buffers, behind the graph state and in front of the stage workspace
struct TrialsBufs {
  int* slot;        // [n][T]
  int* bad;         // [T]
  float* rhs;       // [n][C]: the solves' fp32 right-hand side
  float* x0;        // [n][C]: the initial solve
  float* corr;      // [n][C]: the correction solves
  double* xa;       // [n][C]: the fp64 iterate, ping-pong with xb
  double* xb;
  double* r;        // [n][C]
  double* partial;  // [refine grid x][T l]
  double* colnorm;  // [T l]
  double* scale;
  unsigned* ticket;
  int* round_iters;  // [GLL_LAPLACE_ROUNDS]
};

// base == NULL: size query only
size_t trials_bufs(char* base, int n, int T, int l, TrialsBufs* E) {
  Carver cv(base, ~(size_t)0);
  const size_t nc = (size_t)n * T * padded_classes(l), tl = (size_t)T * l;
  TrialsBufs b;
  b.slot = cv.take<int>((size_t)n * T);
  b.bad = cv.take<int>(T);
  b.rhs = cv.take<float>(nc);
  b.x0 = cv.take<float>(nc);
  b.corr = cv.take<float>(nc);
  b.xa = cv.take<double>(nc);
  b.xb = cv.take<double>(nc);
  b.r = cv.take<double>(nc);
  b.partial = cv.take<double>((size_t)trials_grid(n, T, l).gx * tl);
  b.colnorm = cv.take<double>(tl);
  b.scale = cv.take<double>(1);
  b.ticket = cv.take<unsigned>(1);
  b.round_iters = cv.take<int>(GLL_LAPLACE_ROUNDS);
  if (E) *E = b;
  return align_up(cv.off, 256);
}

// the sizes gll_laplace_eval_trials accepts
bool trials_sizes_ok(int n, int d, int k, int l, int T, int k_lab) {
  if (n < 2 || T < 1 || l < 1 || d < 1 || k_lab < 1 || k_lab >= n) return false;
  if ((long long)n * T * padded_classes(l) > 0x7fffffffLL) return false;
  return k >= 2 && k <= 64 && k <= n && (k <= 33 || n >= 256);
}

// the graph state of the k_lab = 0 stages (a one-column dummy label block, as knn_sym_dist)
int trials_layout(int n, int k, gll_layout* L) { return gll_state_layout(n, k, 1, 0, L); }

// workspace: [graph state | the trials' buffers | stage workspace (kNN, graph stages, CG over C columns)]
size_t trials_ws_bytes(int n, int d, int k, int l, int T) {
  gll_layout L;
  if (trials_layout(n, k, &L)) return 0;
  const size_t stage = std::max(gll_workspace_bytes(n, d, k, 1, 0), cg_ws_bytes(n, T * padded_classes(l)));
  return L.total + trials_bufs(nullptr, n, T, l, nullptr) + stage;
}

int trials_run(const float* X, int n, int d, int k, const void* train_idx, int idx_is_i64, const float* Y, int T, int k_lab, int l,
               int eps_auto, float eps_fixed, float tau, double tol, int cg_max_iter, double* pred, long long* labels,
               const long long* targets, long long* correct_out, double* resid_out, int* info, void* workspace, size_t workspace_bytes,
               cudaStream_t st) {
  const size_t need = trials_ws_bytes(n, d, k, l, T);
  if (workspace_bytes < need) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, need);
    return GLL_ERR_WORKSPACE;
  }
  const int lpad = padded_classes(l), C = T * lpad;
  gll_layout L;
  if (trials_layout(n, k, &L)) return GLL_ERR_ARG;
  char* S = (char*)workspace;
  GraphBufs G = graph_bufs(L, S);
  G.info = info;
  TrialsBufs E;
  const size_t eb = trials_bufs(S + L.total, n, T, l, &E);
  void* ws = S + L.total + eb;
  const size_t ws_bytes = workspace_bytes - L.total - eb;

  GLL_CUDA_CHECK(cudaMemsetAsync(info, 0, sizeof(int) * GLL_INFO_WORDS, st));
  GLL_CUDA_CHECK(cudaMemsetAsync(E.ticket, 0, sizeof(unsigned), st));
  GLL_CUDA_CHECK(cudaMemsetAsync(E.slot, 0xff, sizeof(int) * (size_t)n * T, st));  // -1: not labeled
  GLL_CUDA_CHECK(cudaMemsetAsync(E.bad, 0, sizeof(int) * (size_t)T, st));
  GLL_CUDA_CHECK(cudaMemsetAsync(E.r, 0, sizeof(double) * (size_t)n * C, st));  // padding columns of the right-hand side
  if (correct_out) GLL_CUDA_CHECK(cudaMemsetAsync(correct_out, 0, sizeof(long long) * (size_t)T, st));
  {
    GLL_PROF(KID_LAPLACE_TRIALS_SETUP, st);
    laplace_trials_setup_kernel<<<ceil_div((long long)T * k_lab, 256), 256, 0, st>>>(train_idx, idx_is_i64, n, T, k_lab, E.slot, E.bad,
                                                                                    info);
    GLL_LAUNCH_CHECK();
  }
  int rc = knn_run(X, n, d, k, 0, n, G.knn_idx, G.knn_dist, info, ws, ws_bytes, st);
  if (rc) return rc;
  rc = graph_stages_run(G, nullptr, n, k, 1, 0, eps_auto, eps_fixed, tau, 0, 6, ws, ws_bytes, st);
  if (rc) return rc;

  const TrialsGrid tg = trials_grid(n, T, l);
  TrialsRefineParams P;
  P.row_ptr = G.row_ptr;
  P.col = G.col;
  P.w = G.w;
  P.Y = Y;
  P.slot = E.slot;
  P.bad = E.bad;
  P.r_out = E.r;
  P.partial = E.partial;
  P.colnorm = E.colnorm;
  P.resid = resid_out;
  P.scale = E.scale;
  P.ticket = E.ticket;
  P.info = info;
  P.n = n;
  P.T = T;
  P.k_lab = k_lab;
  P.l = l;
  P.lpad = lpad;
  P.gx = tg.gx;
  P.cw = tg.cw;
  P.tau = (double)tau;
  P.tol = tol;
  const dim3 grid(tg.gx, tg.gy);
  // r = b at x = 0, exactly in fp64: the first solve's right-hand side
  P.x_prev = nullptr;
  P.e = nullptr;
  P.x_out = nullptr;
  P.round = -1;
  {
    GLL_PROF(KID_LAPLACE_REFINE, st);
    laplace_refine_trials_kernel<<<grid, LR_THREADS, 0, st>>>(P);
    GLL_LAUNCH_CHECK();
  }
  unsigned* barrier = (unsigned*)(info + GLL_INFO_CG_BARRIER);
  CgIo io = {E.r, 2, nullptr, 0, nullptr, 0, 0.f, E.slot, T, lpad, 0};
  rc = cg_run(G.uu_ptr, G.uu_col, G.uu_val, G.diag, E.rhs, n, C, -(float)GLL_LAPLACE_CG_RTOL0, cg_max_iter, E.x0,
              info + GLL_INFO_CG_ITERS_FWD, (float*)(info + GLL_INFO_CG_RESID_FWD), nullptr, ws, ws_bytes, st, barrier, &io);
  if (rc) return rc;
  io.rhs_scale = E.scale;
  io.rhs_scale_f64 = 1;
  for (int r = 0; r < GLL_LAPLACE_ROUNDS; ++r) {
    P.x_out = (r % 2 == 0) ? E.xa : E.xb;
    P.x_prev = (r == 0) ? nullptr : (r % 2 == 0 ? E.xb : E.xa);
    P.e = (r == 0) ? E.x0 : E.corr;
    P.round = r;
    {
      GLL_PROF(KID_LAPLACE_REFINE, st);
      laplace_refine_trials_kernel<<<grid, LR_THREADS, 0, st>>>(P);
      GLL_LAUNCH_CHECK();
    }
    rc = cg_run(G.uu_ptr, G.uu_col, G.uu_val, G.diag, E.rhs, n, C, -(float)GLL_LAPLACE_CG_RTOL, cg_max_iter, E.corr, E.round_iters + r,
                nullptr, nullptr, ws, ws_bytes, st, barrier, &io);
    if (rc) return rc;
  }
  {
    GLL_PROF(KID_LAPLACE_FINISH, st);
    laplace_finish_trials_kernel<<<dim3(ceil_div(n, LR_THREADS), T), LR_THREADS, 0, st>>>(
        P.x_out, E.corr, Y, E.slot, E.bad, n, T, k_lab, l, lpad, pred, labels, targets, (unsigned long long*)correct_out, E.scale,
        E.round_iters, GLL_LAPLACE_ROUNDS, info);
    GLL_LAUNCH_CHECK();
  }
  return GLL_OK;
}

}  // namespace
}  // namespace gll

using namespace gll;

extern "C" {

size_t gll_laplace_eval_workspace_bytes(int n, int d, int k, int l, int k_lab) {
  if (n < 2 || l < 1 || k_lab < 1 || k_lab >= n) return 0;
  return eval_ws_bytes(1, n, d, k, l, k_lab);
}

int gll_laplace_eval(const float* X, const float* Y, int n, int d, int k, int l, int k_lab, int eps_auto, float eps_fixed,
                     float tau, double tol, int cg_max_iter, double* pred, long long* labels, const long long* targets,
                     long long* correct_out, int* info, void* workspace, size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(X && Y && pred && labels && info && workspace, "null pointer");
  GLL_REQUIRE(k >= 2 && k <= 64 && (k <= 33 || n >= 256) && k <= n, "k must be in [2, 64] (n >= 256 when k > 33) and <= n");
  GLL_REQUIRE(d >= 1 && l >= 1 && k_lab >= 1 && k_lab < n, "bad sizes");
  GLL_REQUIRE(tol > 0.0 && cg_max_iter >= 1, "tol must be > 0 and cg_max_iter >= 1");
  return eval_run(X, Y, 1, n, d, k, l, k_lab, eps_auto, eps_fixed, tau, tol, cg_max_iter, pred, labels, targets, correct_out, nullptr, info,
                  workspace, workspace_bytes, (cudaStream_t)stream);
}

size_t gll_laplace_eval_batched_workspace_bytes(int B, int n, int d, int k, int l, int k_lab) {
  if (!eval_batched_sizes_ok(B, n, d, k, l, k_lab)) return 0;
  return eval_ws_bytes(B, n, d, k, l, k_lab);
}

int gll_laplace_eval_batched(const float* X, const float* Y, int B, int n, int d, int k, int l, int k_lab, int eps_auto,
                             float eps_fixed, float tau, double tol, int cg_max_iter, double* pred, long long* labels,
                             const long long* targets, long long* correct_out, double* resid_out, int* info, void* workspace,
                             size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(X && Y && pred && labels && info && workspace, "null pointer");
  GLL_REQUIRE(B >= 1 && n >= 1 && (long long)B * n <= 0x7fffffffLL, "need B >= 1 and B n < 2^31");
  GLL_REQUIRE(k >= 2 && k <= 64 && k <= n && (k <= 33 || (long long)B * n >= 256),
              "k must be in [2, 64] and <= n, with B n >= 256 when k > 33");
  GLL_REQUIRE(d >= 1 && l >= 1 && k_lab >= 1 && k_lab < n, "bad sizes");
  GLL_REQUIRE(tol > 0.0 && cg_max_iter >= 1, "tol must be > 0 and cg_max_iter >= 1");
  return eval_run(X, Y, B, n, d, k, l, k_lab, eps_auto, eps_fixed, tau, tol, cg_max_iter, pred, labels, targets, correct_out, resid_out,
                  info, workspace, workspace_bytes, (cudaStream_t)stream);
}

size_t gll_laplace_eval_trials_workspace_bytes(int n, int d, int k, int l, int T, int k_lab) {
  if (!trials_sizes_ok(n, d, k, l, T, k_lab)) return 0;
  return trials_ws_bytes(n, d, k, l, T);
}

int gll_laplace_eval_trials(const float* X, int n, int d, int k, const void* train_idx, int idx_is_i64, const float* Y, int T, int k_lab,
                            int l, int eps_auto, float eps_fixed, float tau, double tol, int cg_max_iter, double* pred,
                            long long* labels, const long long* targets, long long* correct_out, double* resid_out, int* info,
                            void* workspace, size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(X && train_idx && Y && pred && labels && info && workspace, "null pointer");
  GLL_REQUIRE(n >= 2 && T >= 1 && (long long)n * T * padded_classes(l) <= 0x7fffffffLL, "need n >= 2, T >= 1 and n T lpad < 2^31");
  GLL_REQUIRE(k >= 2 && k <= 64 && k <= n && (k <= 33 || n >= 256), "k must be in [2, 64] (n >= 256 when k > 33) and <= n");
  GLL_REQUIRE(d >= 1 && l >= 1 && k_lab >= 1 && k_lab < n, "bad sizes");
  GLL_REQUIRE(tol > 0.0 && cg_max_iter >= 1, "tol must be > 0 and cg_max_iter >= 1");
  return trials_run(X, n, d, k, train_idx, idx_is_i64, Y, T, k_lab, l, eps_auto, eps_fixed, tau, tol, cg_max_iter, pred, labels, targets,
                    correct_out, resid_out, info, workspace, workspace_bytes, (cudaStream_t)stream);
}

}  // extern "C"
