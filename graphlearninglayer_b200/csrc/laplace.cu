// Laplace-learning evaluation on the device (utils.py:570-593 `laplace`, used by test_GL_NP at utils.py:637-660):
// features -> graph -> harmonic extension refined in fp64 to the reference's stop rule -> argmax labels and a hit count.
//
//   gll_laplace_eval(_batched):  K1 + K2/K3 (gll_forward's stages with the caller's k; B graphs: the segmented search)
//                                fp32 Jacobi-CG  (L_uu + tau I) x0 = -L_ul Y,  relative tolerance GLL_LAPLACE_CG_RTOL0
//                                GLL_LAPLACE_ROUNDS x { laplace_refine ; fp32 correction CG at GLL_LAPLACE_CG_RTOL }
//                                laplace_finish
//   gll_laplace_eval_trials:     the same on one graph built with k_lab = 0, T labeled sets masked into one full-graph system;
//                                the first right-hand side is laplace_refine's x = 0 pass
//
// Both solves are R row groups x T column groups of l class columns: B graphs are R = B, T = 1 (UnionRows), the trials R = 1 and
// T trials (TrialRows).  laplace_refine and laplace_finish are written once over those two policies, which say only where a row
// and its columns live, whether a row is clamped in a column group, and what a neighbour's value is.
//
// laplace_refine (round r) reads x_{r-1} (fp64) and the previous fp32 correction e_{r-1}, and writes x_r = x_{r-1} + e_{r-1}
// to the OTHER fp64 buffer (neighbour rows are read while rows are written, so the rounds ping-pong between two buffers).  In
// the same pass it forms the fp64 residual over the full-graph CSR,
//     r_i = sum_j w_ij (u_j - x_i) - tau x_i,   u_j = the label row of a clamped neighbour, else x_r,
// i.e. b - A x with A = D - W_uu + tau I, D = ROW sums of the stored fp32 weights accumulated in fp64, and the reference's
// stop quantity per class column ||M r_c||_2 = sqrt(sum_i r_ic^2 / (D_i + tau + 1e-10)) (make_golden_eval.py:41-45) over the
// rows of one row group.  Per-CTA column partials are added in CTA order by the last CTA of the row group (integer ticket), which
// writes each column group's largest norm; the last row group takes the maximum over the valid column groups and writes the
// correction solve's right-hand-side scale: 1 while some column is above tol, else 0 -- a zero right-hand side stops every CG
// kernel at iteration 0 and the correction is exactly zero, so the round count is fixed and no host decision is needed.  No
// floating-point atomics.  laplace_finish adds the last correction, writes pred, the argmax labels and the hit counts.
#include <algorithm>

#include "cg_common.cuh"
#include "common.cuh"

namespace gll {
namespace {

constexpr int LR_THREADS = 256;

// What laplace_refine and laplace_finish read and write.  `rows` rows per row group; round < 0: r = b only (x = 0), no stop-rule
// bookkeeping.
struct LaplaceParams {
  const int* row_ptr;  // full-graph CSR
  const int* col;
  const float* w;
  const float* Y;        // label rows: k_lab x l (trials: T x k_lab x l)
  const int* slot;       // trials: [n][T], the row's index among trial t's label rows, else -1
  const int* bad;        // [T], or NULL when no column group can be invalid
  const double* x_prev;  // the iterate of the round before, or NULL
  const float* e;        // the fp32 correction (round 0: the first solve), or NULL: x = 0
  double* x_out;         // the iterate of this round (finish: of the last round), or NULL
  double* r_out;         // the next solve's right-hand side
  double* partial;       // [R gx][T l]
  double* colnorm;       // [R][T l]
  double* gmax;          // [R T] with stride gs: the largest column norm of (row group, column group); NaN: a column is not
                         // finite, or the group is invalid.  The trials keep it in colnorm, over each group's first column
  double* resid;         // [R T] or NULL: the caller's copy of gmax
  double* scale;         // 1 scalar
  unsigned* ticket;      // [R + 1]: CTAs done per row group, then row groups done
  int* round_iters;      // [GLL_LAPLACE_ROUNDS]
  int* info;
  double* pred;                 // (T, R rows, l)
  long long* labels;            // (T, R rows)
  const long long* targets;     // [R rows] or NULL
  unsigned long long* correct;  // [R T] or NULL
  int R, rows, T, l, lp, k_lab, gx, cw, fb, gs, round;
  double tau, tol;
};

__device__ __forceinline__ bool group_valid(const LaplaceParams& P, int t) { return P.bad == nullptr || __ldg(P.bad + t) == 0; }

// B graphs as one union: row group g is graph g, whose unlabeled rows are [g mb, (g + 1) mb) of the m = B mb.  The union's CSR
// puts its k_lab = B k_lab labeled rows first, so row i is CSR row k_lab + i and a neighbour j < k_lab is label row j.  x and r
// are [m][l], e [m][lp] and never NULL; no row is clamped.  The policy is built for one column c of the l.
struct UnionRows {
  const LaplaceParams& P;
  const int t = 0, c;
  __device__ UnionRows(const LaplaceParams& P, int c) : P(P), c(c) {}
  __device__ int csr(int i) const { return P.k_lab + i; }
  __device__ size_t xo(int i) const { return (size_t)i * P.l + c; }
  __device__ size_t eo(int i) const { return (size_t)i * P.lp + c; }
  __device__ int slot(int) const { return -1; }
  __device__ const float* yrow(int s) const { return P.Y + (size_t)s * P.l + c; }
  __device__ double x(int i) const { return (P.x_prev ? __ldg(P.x_prev + xo(i)) : 0.0) + (double)__ldg(P.e + eo(i)); }
  __device__ double u(int j) const { return j < P.k_lab ? (double)__ldg(yrow(j)) : x(j - P.k_lab); }
};

// T trials on one graph: one row group of all n rows (row i is CSR row i); column c of the T l is class cl of trial t, column
// t lpad + cl of the C = T lpad columns of x, e and r.  Row i is clamped in trial t when slot[i T + t] >= 0, and a clamped
// neighbour reads its label row Y[t, slot].  x_prev and e may be NULL (x = 0).
struct TrialRows {
  const LaplaceParams& P;
  const int t, cl;
  const size_t C, sc;
  __device__ TrialRows(const LaplaceParams& P, int c)
      : P(P), t(c / P.l), cl(c - t * P.l), C((size_t)P.T * P.lp), sc((size_t)t * P.lp + cl) {}
  __device__ int csr(int i) const { return i; }
  __device__ size_t xo(int i) const { return (size_t)i * C + sc; }
  __device__ size_t eo(int i) const { return xo(i); }
  __device__ int slot(int i) const { return __ldg(P.slot + (size_t)i * P.T + t); }
  __device__ const float* yrow(int s) const { return P.Y + ((size_t)t * P.k_lab + s) * P.l + cl; }
  __device__ double x(int i) const {
    return (P.x_prev ? __ldg(P.x_prev + xo(i)) : 0.0) + (P.e ? (double)__ldg(P.e + eo(i)) : 0.0);
  }
  __device__ double u(int j) const {
    const int s = slot(j);
    return s >= 0 ? (double)__ldg(yrow(s)) : x(j);
  }
};

// Block = RL row lanes x CW columns of the T l (CW = min(T l, 32)); blockIdx.x = g gx + (CTA of row group g), blockIdx.y picks a
// chunk of CW columns.  A thread walks the rows of its lane in row group g in a fixed order and keeps its own partial sum of
// r^2 / diag: the reduction order depends on nothing but the launch shape.  A row clamped in the column's group, and every row of
// an invalid group, has r = 0.
template <class Rows>
__global__ void __launch_bounds__(LR_THREADS) laplace_refine_kernel(LaplaceParams P) {
  __shared__ double red[LR_THREADS];
  __shared__ bool last;
  const int cw = P.cw, rl_count = LR_THREADS / cw, TL = P.T * P.l;
  const int tid = threadIdx.x, rl = tid / cw, cc = tid - rl * cw;
  const int c = blockIdx.y * cw + cc;
  const int g = blockIdx.x / P.gx, bx = blockIdx.x - g * P.gx;
  double acc = 0.0;
  if (rl < rl_count && c < TL) {
    const int i_end = (g + 1) * P.rows;
    const Rows rows(P, c);
    const bool valid = group_valid(P, rows.t);
    for (int i = g * P.rows + bx * rl_count + rl; i < i_end; i += P.gx * rl_count) {
      const size_t o = rows.xo(i);
      const double xi = rows.x(i);
      if (P.x_out) P.x_out[o] = xi;
      if (!valid || rows.slot(i) >= 0) {
        P.r_out[o] = 0.0;
        continue;
      }
      const int a = rows.csr(i), e1 = __ldg(P.row_ptr + a + 1);
      double s = 0.0, deg = 0.0;
      for (int e = __ldg(P.row_ptr + a); e < e1; ++e) {
        const int j = __ldg(P.col + e);
        const double wv = (double)__ldg(P.w + e);
        s = fma(wv, rows.u(j) - xi, s);
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
    double s = 0.0;
    for (int q = 0; q < rl_count; ++q) s += red[q * cw + tid];
    P.partial[(size_t)blockIdx.x * TL + c] = s;
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) last = atomicAdd(P.ticket + g, 1u) == P.gx * gridDim.y - 1u;
  __syncthreads();
  if (!last) return;
  __threadfence();
  // the last CTA of row group g: its column norms, partials added in CTA order
  const int lane = tid & 31, warp = tid >> 5;
  const double* part = P.partial + (size_t)g * P.gx * TL;
  double* colnorm = P.colnorm + (size_t)g * TL;
  for (int c2 = warp; c2 < TL; c2 += LR_THREADS / 32) {
    double s = 0.0;
    for (int q = lane; q < P.gx; q += 32) s += __ldcg(part + (size_t)q * TL + c2);
    s = warp_sum(s);
    if (lane == 0) colnorm[c2] = sqrt(s);
  }
  __syncthreads();
  for (int t = tid; t < P.T; t += LR_THREADS) {
    double mx = 0.0;
    bool bad = !group_valid(P, t);
    for (int c2 = t * P.l; c2 < (t + 1) * P.l; ++c2) {
      const double v = colnorm[c2];
      if (!(v == v) || isinf(v)) bad = true;
      mx = fmax(mx, v);
    }
    const double gv = bad ? __longlong_as_double(0x7ff8000000000000LL) : mx;
    P.gmax[((size_t)g * P.T + t) * P.gs] = gv;  // over colnorm[t l] when gmax is colnorm: only this thread read it
    if (P.resid != nullptr) P.resid[(size_t)g * P.T + t] = gv;
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    P.ticket[g] = 0u;  // rewound for the next round
    last = atomicAdd(P.ticket + P.R, 1u) == (unsigned)P.R - 1u;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  // the last row group: the maximum over the valid groups is exact, so the order of the reduction does not matter
  double mx = 0.0;
  bool bad = false;
  for (int q = tid; q < P.R * P.T; q += LR_THREADS) {
    if (!group_valid(P, q % P.T)) continue;
    const double v = __ldcg(P.gmax + (size_t)q * P.gs);
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
    P.ticket[P.R] = 0u;
  }
}

// Thread per (row, group): group q = (row group g, column group t) = (q / T, q % T) owns the fb CTAs [q fb, (q + 1) fb).  pred =
// x + e, or the label row where the row is clamped, or NaN for an invalid group; labels = first maximal column (-1 for an invalid
// group); hits of the unclamped rows counted with one integer atomic per CTA into correct[q] (-1 for an invalid group).  CTA 0
// also writes the correction-CG iteration counts and the convergence status.
template <class Rows>
__global__ void __launch_bounds__(LR_THREADS) laplace_finish_kernel(LaplaceParams P) {
  __shared__ int part[LR_THREADS / 32];
  const int q = blockIdx.x / P.fb, g = q / P.T, t = q - g * P.T, li = (blockIdx.x - q * P.fb) * LR_THREADS + threadIdx.x;
  const bool valid = group_valid(P, t);
  int hit = 0;
  if (li < P.rows) {
    const Rows rows(P, t * P.l);  // the group's first column: its l columns follow it in x, e and Y
    const int i = g * P.rows + li;
    const size_t oi = (size_t)t * P.R * P.rows + i;
    double* p = P.pred + oi * P.l;
    long long arg = -1;
    if (!valid) {
      for (int c = 0; c < P.l; ++c) p[c] = __longlong_as_double(0x7ff8000000000000LL);
    } else {
      const int s = rows.slot(i);
      const size_t xo = rows.xo(i), eo = rows.eo(i);
      double best = 0.0;
      for (int c = 0; c < P.l; ++c) {
        const double v = (s >= 0) ? (double)__ldg(rows.yrow(s) + c) : P.x_out[xo + c] + (double)__ldg(P.e + eo + c);
        p[c] = v;
        if (c == 0 || v > best) {
          best = v;
          arg = c;
        }
      }
      if (s < 0 && P.targets != nullptr) {
        const long long tg = __ldg(P.targets + i);
        hit = (tg >= 0 && tg == arg) ? 1 : 0;
      }
    }
    P.labels[oi] = arg;
  }
  if (P.correct != nullptr) {
    hit = warp_sum(hit);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = hit;
    __syncthreads();
    if (threadIdx.x == 0) {
      int s = 0;
      for (int w = 0; w < LR_THREADS / 32; ++w) s += part[w];
      if (!valid) {
        if (blockIdx.x == q * P.fb) P.correct[q] = ~0ull;  // -1; no other CTA of an invalid group adds anything
      } else if (s) {
        atomicAdd(P.correct + q, (unsigned long long)s);
      }
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    int tot = 0;
    unsigned packed[2] = {0u, 0u};
    for (int r = 0; r < GLL_LAPLACE_ROUNDS; ++r) {
      const int it = P.round_iters[r];
      tot += it;
      if (r < 4) packed[r >> 1] |= (unsigned)min(it, 65535) << (16 * (r & 1));
    }
    P.info[GLL_INFO_LAPLACE_CG_ITERS] = tot;
    P.info[GLL_INFO_LAPLACE_ROUND_ITERS] = (int)packed[0];
    P.info[GLL_INFO_LAPLACE_ROUND_ITERS + 1] = (int)packed[1];
    if (*P.scale != 0.0) atomicOr(P.info + GLL_INFO_STATUS, GLL_STATUS_CG_NOT_CONVERGED);  // tol unmet after the last round
  }
}

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

// Launch shape of laplace_refine over `cols` columns and row groups of `rows` rows: cw columns per CTA, gy column chunks, gx CTAs
// per row group, at most 4 per SM (spread: about 4 per SM over all chunks, so the last CTA of the trials adds few partials per
// column).  The shape fixes the order of the column sums, and with it the bits of resid.
struct RefineGrid {
  int cw, gy, gx;
};
RefineGrid refine_grid(int rows, int cols, bool spread) {
  const int cw = min(cols, 32), gy = ceil_div(cols, cw), ctas = 4 * device_info().sms;
  return {cw, gy, max(1, min(ceil_div(rows, LR_THREADS / cw), spread ? ceil_div(ctas, gy) : ctas))};
}

// The evaluation's own buffers, behind the graph state and in front of the stage workspace.  The trials add the slot table, bad,
// an fp32 right-hand side, first solution and correction of C = T lpad columns (B graphs use the graph state's) and a second fp64
// iterate (B graphs ping-pong with the caller's pred).
struct EvalBufs {
  int* slot;  // [n][T]
  int* bad;   // [T]
  float* rhs;
  float* x0;
  float* corr;
  double* xb;
  double* xa;       // fp64 iterate: [n][C] (B graphs: [m][l])
  double* r;        // as xa
  double* partial;  // [R gx][T l]
  double* colnorm;  // [R][T l]
  double* gmax;     // [R] (trials: colnorm, stride l)
  double* scale;
  unsigned* ticket;  // [R + 1]
  int* round_iters;  // [GLL_LAPLACE_ROUNDS]
};

// base == NULL: size query only
size_t eval_bufs(char* base, int R, int rows, int T, int l, bool trials, EvalBufs* E) {
  Carver cv(base, ~(size_t)0);
  const size_t N = (size_t)R * rows, tl = (size_t)T * l, nx = trials ? N * T * padded_classes(l) : N * l;
  EvalBufs b = {};
  if (trials) {
    b.slot = cv.take<int>(N * T);
    b.bad = cv.take<int>(T);
    b.rhs = cv.take<float>(nx);
    b.x0 = cv.take<float>(nx);
    b.corr = cv.take<float>(nx);
    b.xb = cv.take<double>(nx);
  }
  b.xa = cv.take<double>(nx);
  b.r = cv.take<double>(nx);
  b.partial = cv.take<double>((size_t)R * refine_grid(rows, T * l, trials).gx * tl);
  b.colnorm = cv.take<double>(R * tl);
  b.gmax = trials ? b.colnorm : cv.take<double>(R);
  b.scale = cv.take<double>(1);
  b.ticket = cv.take<unsigned>((size_t)R + 1);
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
  return L.total + eval_bufs(nullptr, B, n - k_lab, 1, l, false, nullptr) + stage;
}

// the graph state of the trials' k_lab = 0 stages (a one-column dummy label block, as knn_sym_dist)
int trials_layout(int n, int k, gll_layout* L) { return gll_state_layout(n, k, 1, 0, L); }

// workspace of T trials: [graph state | the evaluation's buffers | stage workspace (kNN, graph stages, CG over C columns)]
size_t trials_ws_bytes(int n, int d, int k, int l, int T) {
  gll_layout L;
  if (trials_layout(n, k, &L)) return 0;
  const size_t stage = std::max(gll_workspace_bytes(n, d, k, 1, 0), cg_ws_bytes(n, T * padded_classes(l)));
  return L.total + eval_bufs(nullptr, 1, n, T, l, true, nullptr) + stage;
}

// a run's carved workspace; P holds what both kernels read, the rounds fill in the iterates
struct Run {
  GraphBufs G;
  EvalBufs E;
  LaplaceParams P;
  void* ws;  // stage workspace
  size_t ws_bytes;
};

// Checks and carves the workspace [graph state | the evaluation's buffers | stage workspace] of a run that needs `need` bytes,
// zeroes info, the tickets and the hit counts, and fills the kernels' parameters.
int begin_run(const gll_layout& L, size_t need, bool trials, int R, int rows, int T, int l, int k_lab, const float* Y, float tau,
              double tol, double* pred, long long* labels, const long long* targets, long long* correct_out, double* resid_out,
              int* info, void* workspace, size_t workspace_bytes, cudaStream_t st, Run* run) {
  if (workspace_bytes < need) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, need);
    return GLL_ERR_WORKSPACE;
  }
  char* S = (char*)workspace;
  Run& u = *run;
  u.G = graph_bufs(L, S);
  u.G.info = info;  // the caller's info block in place of the state's
  const size_t eb = eval_bufs(S + L.total, R, rows, T, l, trials, &u.E);
  u.ws = S + L.total + eb;
  u.ws_bytes = workspace_bytes - L.total - eb;
  GLL_CUDA_CHECK(cudaMemsetAsync(info, 0, sizeof(int) * GLL_INFO_WORDS, st));
  GLL_CUDA_CHECK(cudaMemsetAsync(u.E.ticket, 0, sizeof(unsigned) * ((size_t)R + 1), st));
  if (correct_out) GLL_CUDA_CHECK(cudaMemsetAsync(correct_out, 0, sizeof(long long) * (size_t)R * T, st));
  const RefineGrid rg = refine_grid(rows, T * l, trials);
  LaplaceParams& P = u.P;
  P = LaplaceParams{};
  P.row_ptr = u.G.row_ptr;
  P.col = u.G.col;
  P.w = u.G.w;
  P.Y = Y;
  P.slot = u.E.slot;
  P.bad = u.E.bad;
  P.r_out = u.E.r;
  P.partial = u.E.partial;
  P.colnorm = u.E.colnorm;
  P.gmax = u.E.gmax;
  P.gs = trials ? l : 1;
  P.resid = resid_out;
  P.scale = u.E.scale;
  P.ticket = u.E.ticket;
  P.round_iters = u.E.round_iters;
  P.info = info;
  P.pred = pred;
  P.labels = labels;
  P.targets = targets;
  P.correct = (unsigned long long*)correct_out;
  P.R = R;
  P.rows = rows;
  P.T = T;
  P.l = l;
  P.lp = padded_classes(l);
  P.k_lab = k_lab;
  P.gx = rg.gx;
  P.cw = rg.cw;
  P.fb = ceil_div(rows, LR_THREADS);
  P.tau = (double)tau;
  P.tol = tol;
  return GLL_OK;
}

template <class Rows>
int launch_refine(const LaplaceParams& P, cudaStream_t st) {
  GLL_PROF(KID_LAPLACE_REFINE, st);
  laplace_refine_kernel<Rows><<<dim3(P.R * P.gx, ceil_div(P.T * P.l, P.cw)), LR_THREADS, 0, st>>>(P);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

// The rounds after the first solve, and the finish.  Round r refines x0 (r = 0) or the iterate of round r - 1 plus corr, and writes
// `fin` when (GLL_LAPLACE_ROUNDS - 1 - r) is even, `other` otherwise, so the last round writes `fin`; correction(iters) then
// solves for corr.
template <class Rows, class Correction>
int refine_rounds(LaplaceParams P, const float* x0, const float* corr, double* fin, double* other, Correction correction,
                  cudaStream_t st) {
  for (int r = 0; r < GLL_LAPLACE_ROUNDS; ++r) {
    const bool to_fin = (GLL_LAPLACE_ROUNDS - 1 - r) % 2 == 0;
    P.x_prev = (r == 0) ? nullptr : (to_fin ? other : fin);
    P.x_out = to_fin ? fin : other;
    P.e = (r == 0) ? x0 : corr;
    P.round = r;
    int rc = launch_refine<Rows>(P, st);
    if (rc) return rc;
    rc = correction(P.round_iters + r);
    if (rc) return rc;
  }
  GLL_PROF(KID_LAPLACE_FINISH, st);
  laplace_finish_kernel<Rows><<<P.R * P.T * P.fb, LR_THREADS, 0, st>>>(P);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

// gll_laplace_eval (B = 1) and gll_laplace_eval_batched: sizes are checked by the callers
int eval_run(const float* X, const float* Y, int B, int n, int d, int k, int l, int k_lab, int eps_auto, float eps_fixed, float tau,
             double tol, int cg_max_iter, double* pred, long long* labels, const long long* targets, long long* correct_out,
             double* resid_out, int* info, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const int N = B * n, K = B * k_lab, m = N - K;
  gll_layout L;
  if (gll_state_layout(N, k, l, K, &L)) return GLL_ERR_ARG;
  Run u;
  int rc = begin_run(L, eval_ws_bytes(B, n, d, k, l, k_lab), false, B, n - k_lab, 1, l, K, Y, tau, tol, pred, labels, targets,
                     correct_out, resid_out, info, workspace, workspace_bytes, st, &u);
  if (rc) return rc;
  const GraphBufs& G = u.G;
  rc = (B == 1) ? knn_run(X, n, d, k, 0, n, G.knn_idx, G.knn_dist, info, u.ws, u.ws_bytes, st)
                : batched_knn_run(X, B, n, d, k, k_lab, G, u.ws, u.ws_bytes, st);
  if (rc) return rc;
  rc = graph_stages_run(G, Y, N, k, l, K, eps_auto, eps_fixed, tau, 0, 6, u.ws, u.ws_bytes, st);
  if (rc) return rc;
  float* x0 = G.ut + (size_t)K * u.P.lp;
  float* corr = G.wt;  // the adjoint's region, free in an evaluation
  // No sparsity hint (0): the evaluation system is never routed to the cluster kernel.  No status pointer either: an inner solve
  // that stops at the fp32 floor is not a failure -- the fp64 rounds decide convergence.  B graphs are one block-diagonal system:
  // every CG solves them together, with step lengths shared by the graphs (per class column).
  CgSolve S = cg_system(G, m, l, -(float)GLL_LAPLACE_CG_RTOL0, cg_max_iter);
  S.x = x0;
  S.iters_out = info + GLL_INFO_CG_ITERS_FWD;
  S.resid_out = (float*)(info + GLL_INFO_CG_RESID_FWD);
  rc = cg_run(S, u.ws, u.ws_bytes, st);
  if (rc) return rc;
  CgSolve R = S;  // the correction of a refinement round
  R.x = corr;
  R.tol = -(float)GLL_LAPLACE_CG_RTOL;
  R.resid_out = nullptr;
  R.rhs_src = u.E.r;
  R.rhs_kind = 2;
  R.rhs_scale = u.E.scale;
  R.rhs_scale_f64 = 1;
  return refine_rounds<UnionRows>(u.P, x0, corr, pred, u.E.xa, [&](int* iters) {
    R.iters_out = iters;
    return cg_run(R, u.ws, u.ws_bytes, st);
  }, st);
}

// gll_laplace_eval_trials: trial t clamps the k_lab rows train_idx[t] to the label rows Y[t] and solves the other rows.  The graph
// is the same in every trial, so the stages run once with k_lab = 0: the system is the FULL graph A = D + tau I - W over all n
// rows, and trial t masks its clamped rows out of its own columns (cg_persistent_kernel<true>: A p is zeroed there, so r, p and
// x stay 0 on those rows).  Every [n][C] array has C = T lpad columns, lpad = padded_classes(l): trial t owns the columns
// [t lpad, t lpad + l), so a class quad never spans two trials.  slot[i T + t] = s when train_idx[t, s] == i, else -1.
int trials_run(const float* X, int n, int d, int k, const void* train_idx, int idx_is_i64, const float* Y, int T, int k_lab, int l,
               int eps_auto, float eps_fixed, float tau, double tol, int cg_max_iter, double* pred, long long* labels,
               const long long* targets, long long* correct_out, double* resid_out, int* info, void* workspace, size_t workspace_bytes,
               cudaStream_t st) {
  gll_layout L;
  if (trials_layout(n, k, &L)) return GLL_ERR_ARG;
  Run u;
  int rc = begin_run(L, trials_ws_bytes(n, d, k, l, T), true, 1, n, T, l, k_lab, Y, tau, tol, pred, labels, targets, correct_out,
                     resid_out, info, workspace, workspace_bytes, st, &u);
  if (rc) return rc;
  const GraphBufs& G = u.G;
  const EvalBufs& E = u.E;
  const int C = T * u.P.lp;
  GLL_CUDA_CHECK(cudaMemsetAsync(E.slot, 0xff, sizeof(int) * (size_t)n * T, st));  // -1: not labeled
  GLL_CUDA_CHECK(cudaMemsetAsync(E.bad, 0, sizeof(int) * (size_t)T, st));
  GLL_CUDA_CHECK(cudaMemsetAsync(E.r, 0, sizeof(double) * (size_t)n * C, st));  // padding columns of the right-hand side
  {
    GLL_PROF(KID_LAPLACE_TRIALS_SETUP, st);
    laplace_trials_setup_kernel<<<ceil_div((long long)T * k_lab, 256), 256, 0, st>>>(train_idx, idx_is_i64, n, T, k_lab, E.slot, E.bad,
                                                                                    info);
    GLL_LAUNCH_CHECK();
  }
  rc = knn_run(X, n, d, k, 0, n, G.knn_idx, G.knn_dist, info, u.ws, u.ws_bytes, st);
  if (rc) return rc;
  rc = graph_stages_run(G, nullptr, n, k, 1, 0, eps_auto, eps_fixed, tau, 0, 6, u.ws, u.ws_bytes, st);
  if (rc) return rc;
  LaplaceParams P0 = u.P;  // r = b at x = 0, exactly in fp64: the first solve's right-hand side
  P0.round = -1;
  rc = launch_refine<TrialRows>(P0, st);
  if (rc) return rc;
  CgSolve S = cg_system(G, n, C, -(float)GLL_LAPLACE_CG_RTOL0, cg_max_iter);
  S.rhs = E.rhs;
  S.x = E.x0;
  S.iters_out = info + GLL_INFO_CG_ITERS_FWD;
  S.resid_out = (float*)(info + GLL_INFO_CG_RESID_FWD);
  S.rhs_src = E.r;
  S.rhs_kind = 2;
  S.mask_slot = E.slot;
  S.mask_trials = T;
  S.mask_cols = u.P.lp;
  rc = cg_run(S, u.ws, u.ws_bytes, st);
  if (rc) return rc;
  CgSolve R = S;  // the correction of a refinement round
  R.x = E.corr;
  R.tol = -(float)GLL_LAPLACE_CG_RTOL;
  R.resid_out = nullptr;
  R.rhs_scale = E.scale;
  R.rhs_scale_f64 = 1;
  return refine_rounds<TrialRows>(u.P, E.x0, E.corr, E.xb, E.xa, [&](int* iters) {
    R.iters_out = iters;
    return cg_run(R, u.ws, u.ws_bytes, st);
  }, st);
}

// The first size rule a shape breaks, in GLL_REQUIRE's wording, or NULL.  The workspace queries and the entry points share them.
#define SIZE_RULE(cond, msg) \
  if (!(cond)) return msg " (" #cond ")"

const char* batched_sizes_error(int B, int n, int d, int k, int l, int k_lab) {
  SIZE_RULE(B >= 1 && n >= 1 && (long long)B * n <= 0x7fffffffLL, "need B >= 1 and B n < 2^31");
  SIZE_RULE(k >= 2 && k <= 64 && k <= n && (k <= 33 || (long long)B * n >= 256),
            "k must be in [2, 64] and <= n, with B n >= 256 when k > 33");
  SIZE_RULE(d >= 1 && l >= 1 && k_lab >= 1 && k_lab < n, "bad sizes");
  return nullptr;
}

const char* trials_sizes_error(int n, int d, int k, int l, int T, int k_lab) {
  SIZE_RULE(n >= 2 && T >= 1 && (long long)n * T * padded_classes(l) <= 0x7fffffffLL, "need n >= 2, T >= 1 and n T lpad < 2^31");
  SIZE_RULE(k >= 2 && k <= 64 && k <= n && (k <= 33 || n >= 256), "k must be in [2, 64] (n >= 256 when k > 33) and <= n");
  SIZE_RULE(d >= 1 && l >= 1 && k_lab >= 1 && k_lab < n, "bad sizes");
  // laplace_refine puts ceil(T l / 32) column chunks in gridDim.y, which stops at 65535
  SIZE_RULE((long long)T * l <= 65535LL * 32, "need T l <= 2097120");
  return nullptr;
}

int refuse(const char* why) {
  set_error("%s", why);
  return GLL_ERR_ARG;
}

}  // namespace
}  // namespace gll

using namespace gll;

extern "C" {

// The one-graph query has always sized any k and d the stages can size, so it checks only the label split; the entry point's
// rules are the ones its GLL_REQUIRE chain states.
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
  return batched_sizes_error(B, n, d, k, l, k_lab) ? 0 : eval_ws_bytes(B, n, d, k, l, k_lab);
}

int gll_laplace_eval_batched(const float* X, const float* Y, int B, int n, int d, int k, int l, int k_lab, int eps_auto,
                             float eps_fixed, float tau, double tol, int cg_max_iter, double* pred, long long* labels,
                             const long long* targets, long long* correct_out, double* resid_out, int* info, void* workspace,
                             size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(X && Y && pred && labels && info && workspace, "null pointer");
  if (const char* why = batched_sizes_error(B, n, d, k, l, k_lab)) return refuse(why);
  GLL_REQUIRE(tol > 0.0 && cg_max_iter >= 1, "tol must be > 0 and cg_max_iter >= 1");
  return eval_run(X, Y, B, n, d, k, l, k_lab, eps_auto, eps_fixed, tau, tol, cg_max_iter, pred, labels, targets, correct_out, resid_out,
                  info, workspace, workspace_bytes, (cudaStream_t)stream);
}

size_t gll_laplace_eval_trials_workspace_bytes(int n, int d, int k, int l, int T, int k_lab) {
  return trials_sizes_error(n, d, k, l, T, k_lab) ? 0 : trials_ws_bytes(n, d, k, l, T);
}

int gll_laplace_eval_trials(const float* X, int n, int d, int k, const void* train_idx, int idx_is_i64, const float* Y, int T, int k_lab,
                            int l, int eps_auto, float eps_fixed, float tau, double tol, int cg_max_iter, double* pred,
                            long long* labels, const long long* targets, long long* correct_out, double* resid_out, int* info,
                            void* workspace, size_t workspace_bytes, void* stream) {
  GLL_REQUIRE(X && train_idx && Y && pred && labels && info && workspace, "null pointer");
  if (const char* why = trials_sizes_error(n, d, k, l, T, k_lab)) return refuse(why);
  GLL_REQUIRE(tol > 0.0 && cg_max_iter >= 1, "tol must be > 0 and cg_max_iter >= 1");
  return trials_run(X, n, d, k, train_idx, idx_is_i64, Y, T, k_lab, l, eps_auto, eps_fixed, tau, tol, cg_max_iter, pred, labels, targets,
                    correct_out, resid_out, info, workspace, workspace_bytes, (cudaStream_t)stream);
}

}  // extern "C"
