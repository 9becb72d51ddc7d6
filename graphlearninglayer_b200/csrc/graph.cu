// K2 + K3 -- the symmetrised kNN graph as a CSR with sorted rows, bandwidths, edge weights, degree and the linear system
// of the unlabeled block, as ONE persistent cooperative kernel.
//
//   K2 (GLL.py:192-198: coo -> csr, D + D^T.*(D^T > D) - D.*(D^T > D), sparse.find).  Distances are bit-symmetric (knn.cu
//      computes d_ij and d_ji identically), so the elementwise max reduces to the UNION of the directed kNN edges; exact
//      zeros (self, duplicate points) are not edges because sparse.find drops them.
//   K3 eps_i : GLL.py:205 (auto: distance to the last kNN entry kappa(i)) / GLL.py:226 (fixed)
//      W_ij  : GLL.py:216 / 233   exp(-4 d^2 / eps_i / eps_j), evaluated in fp64, stored fp32
//      deg_i : GLL.py:29          csgraph.laplacian degree (sum of the stored fp32 weights, so L 1 = 0 holds)
//      L_uu  : GLL.py:37,48       kept as diag = deg + tau and a compact CSR of the off-diagonal weights
//      rhs   : GLL.py:53          -L_ul Y = W_ul Y
//      The dense n x n matrix C of GLL.py:209-213 is replaced by the map kappa[n].
//
// Phases, separated by grid barriers (one atomic counter, ~1.2 us each with 148 CTAs -- tools/xchg_bench.cu):
//   0 count     per kNN entry: edge or not, listed by both ends or only by i (then the reverse edge j -> i is created)
//   1 scan      row lengths -> row_ptr (per-CTA tile scan, barrier, tile offsets)
//   2 fill      forward edges at deterministic slots, reverse edges through an integer cursor
//   3 rows      warp per row: rank sort by column (removes the only order nondeterminism), then -- same warp, same row --
//               eps, kappa, W, degree, diag, rhs and the count of unlabeled neighbours
//   4 scan      unlabeled-neighbour counts -> uu_ptr
//   5 uu fill   compact off-diagonal CSR of L_uu
// Round 1 ran these as seven launches of 7-18 us each (4.6 MB of data: a microsecond of traffic apiece); the time was
// launch latency and tails, 0.085 ms of the 0.54 ms step at C2.
#include <math.h>
#include <string.h>

#include "cg_common.cuh"
#include "common.cuh"

namespace gll {
namespace {

constexpr int GF_THREADS = 1024;

struct GfParams {
  unsigned long long* trace;  // debug timeline (gll_debug_cg_trace buffer): trace[64 + phase] = %globaltimer at the phase's end
  // inputs
  const int* knn_idx;
  const float* knn_dist;
  const float* Y;
  int n, k, l, lp, k_lab, eps_auto;
  float eps_fixed, tau;
  int phase_begin, phase_end;  // [begin, end) of the phases above (the stage entry points run K2 and K3 separately)
  // K2 outputs / scratch
  int* row_ptr;
  int* col;
  float* dist;
  int* len;      // [n + 1] zeroed
  int* cursor;   // [n + 1] zeroed
  int* col_tmp;
  float* dist_tmp;
  unsigned char* flag;
  // K3 outputs / scratch
  float* eps;
  int* kappa;
  float* w;
  float* deg;
  int* uu_cnt;
  int* uu_ptr;
  int* uu_col;
  float* uu_val;
  float* diag;
  float* rhs;
  float* ut;
  int* info;
  int* tile_sums;     // [grid + 1]
  unsigned* counter;  // grid barrier, zeroed
};

__device__ __forceinline__ unsigned gf_ld_acquire(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void gf_barrier(unsigned* counter, unsigned& target) {
  target += gridDim.x;
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(counter), "r"(1u) : "memory");
    while (gf_ld_acquire(counter) < target) {
    }
  }
  __syncthreads();
}

__device__ __forceinline__ int block_exclusive_scan(int v, int* total, int* smem /* [33] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(FULL, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) smem[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int s = (lane < nw) ? smem[lane] : 0;
    int sinc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(FULL, sinc, o);
      if (lane >= o) sinc += t;
    }
    smem[lane] = sinc - s;  // exclusive warp offsets
    if (lane == 31) smem[32] = sinc;
  }
  __syncthreads();
  int res = inc - v + smem[warp];
  *total = smem[32];
  __syncthreads();
  return res;
}

// Grid-wide exclusive scan of in[0..cnt) into out[0..cnt], out[cnt] = total: CTA b scans the tile [b T, (b+1) T) with a running
// carry and publishes the tile total; after a barrier every CTA adds the totals of the tiles before its own.
__device__ void grid_scan(const int* __restrict__ in, int cnt, int* __restrict__ out, int* __restrict__ tile_sums, unsigned* counter,
                          unsigned& target, int* sm) {
  const int G = gridDim.x, b = blockIdx.x;
  const int T = (cnt + G - 1) / G;
  const int lo = min(cnt, b * T), hi = min(cnt, lo + T);
  int carry = 0;
  for (int base = lo; base < hi; base += GF_THREADS * 4) {
    const int i0 = base + threadIdx.x * 4;
    int v[4], s = 0;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      v[t] = (i0 + t < hi) ? in[i0 + t] : 0;
      s += v[t];
    }
    int tot;
    int ex = block_exclusive_scan(s, &tot, sm) + carry;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      if (i0 + t < hi) out[i0 + t] = ex;
      ex += v[t];
    }
    carry += tot;
  }
  if (threadIdx.x == 0) tile_sums[b] = carry;
  gf_barrier(counter, target);
  // offset of my tile = sum of the earlier tiles' totals (G <= a few hundred: one warp)
  if (threadIdx.x < 32) {
    int off = 0, all = 0;
    for (int t = threadIdx.x; t < G; t += 32) {
      const int v = __ldcg(tile_sums + t);
      all += v;
      if (t < b) off += v;
    }
    off = warp_sum(off);
    all = warp_sum(all);
    if (threadIdx.x == 0) {
      sm[0] = off;
      if (b == G - 1) out[cnt] = all;
    }
  }
  __syncthreads();
  const int off = sm[0];
  if (off != 0)
    for (int i = lo + threadIdx.x; i < hi; i += GF_THREADS) out[i] += off;
  __syncthreads();
}

__device__ __forceinline__ bool is_edge(int i, int j, float dd, int n) { return dd > 0.f && j != i && j >= 0 && j < n; }

__global__ void __launch_bounds__(GF_THREADS, 1) graph_weights_kernel(GfParams P) {
  __shared__ int sm[33];
  // debug timeline (tools/graph_trace.py): CTA 0, thread 0, %globaltimer (256 ns steps) at the end of every phase
#define GF_STAMP(slot) do { if (P.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); P.trace[64 + (slot)] = t_; } } while (0)
  GF_STAMP(0);
  const int n = P.n, k = P.k;
  const long long nthreads = (long long)gridDim.x * GF_THREADS, gtid = (long long)blockIdx.x * GF_THREADS + threadIdx.x;
  const long long total = (long long)n * k;
  const int lane = threadIdx.x & 31;
  const long long gwarp = gtid >> 5, nwarps = nthreads >> 5;
  unsigned target = 0;
  int ph = P.phase_begin;

  // ---- 0: warp per row, lane = kNN slot.  flag byte per entry: bits 0-1 = 0 not an edge, 1 edge listed by both ends, 2 edge
  //         listed only by i (the reverse edge j -> i must be created); bits 2-7 = valid entries before it in its row ----
  if (ph == 0 && ph < P.phase_end) {
    for (long long wi = gwarp; wi < n; wi += nwarps) {
      const int i = (int)wi;
      int carry = 0;
      for (int s0 = 0; s0 < k; s0 += 32) {  // k <= 64: at most two rounds
        const int sl = s0 + lane;
        unsigned char f = 0;
        int j = -1;
        if (sl < k) {
          j = P.knn_idx[(size_t)i * k + sl];
          const float dd = P.knn_dist[(size_t)i * k + sl];
          if (is_edge(i, j, dd, n)) {
            // distances are bit-symmetric, so an entry i in row j carries the same non-zero distance: scan the indices only
            bool mutual = false;
            const int* rj = P.knn_idx + (size_t)j * k;
            for (int u = 0; u < k; ++u) mutual |= (__ldg(rj + u) == i);
            if (!mutual) atomicAdd(&P.len[j], 1);
            f = mutual ? 1 : 2;
          }
        }
        const unsigned valid = __ballot_sync(FULL, f != 0);
        const int before = carry + __popc(valid & ((1u << lane) - 1u));
        if (sl < k) P.flag[(size_t)i * k + sl] = (unsigned char)(f | (before << 2));
        carry += __popc(valid);
      }
      if (lane == 0 && carry) atomicAdd(&P.len[i], carry);
    }
    gf_barrier(P.counter, target);
    GF_STAMP(1);
    ++ph;
  }
  // ---- 1: row_ptr ----
  if (ph == 1 && ph < P.phase_end) {
    grid_scan(P.len, n, P.row_ptr, P.tile_sums, P.counter, target, sm);
    gf_barrier(P.counter, target);
    GF_STAMP(2);
    ++ph;
  }
  // ---- 2: forward edges of row i fill the head of the row in kNN order, reverse edges the tail through a cursor ----
  if (ph == 2 && ph < P.phase_end) {
    for (long long t = gtid; t < total; t += nthreads) {
      const unsigned f = P.flag[t];
      if ((f & 3u) == 0) continue;
      const int i = (int)(t / k);
      const int j = P.knn_idx[t];
      const float dd = P.knn_dist[t];
      const int p = __ldcg(P.row_ptr + i) + (int)(f >> 2);
      P.col_tmp[p] = j;
      P.dist_tmp[p] = dd;
      if ((f & 3u) == 2) {
        const int q = __ldcg(P.row_ptr + j + 1) - 1 - atomicAdd(&P.cursor[j], 1);
        P.col_tmp[q] = i;
        P.dist_tmp[q] = dd;
      }
    }
    gf_barrier(P.counter, target);
    GF_STAMP(3);
    ++ph;
  }
  // ---- 3: warp per row: rank sort by column (columns are unique within a row), then the row's weights ----
  if (ph == 3 && ph < P.phase_end) {
    const bool do_sort = P.phase_begin <= 2 || P.col_tmp != nullptr;
    const bool do_weights = P.phase_end > 3 && P.w != nullptr;
    const int l = P.l, lp = P.lp, k_lab = P.k_lab;
    if (gtid == 0 && P.info != nullptr && do_sort) P.info[GLL_INFO_NNZ] = __ldcg(P.row_ptr + n);
    for (long long wi = gwarp; wi < n; wi += nwarps) {
      const int i = (int)wi;
      const int e0 = __ldcg(P.row_ptr + i), e1 = __ldcg(P.row_ptr + i + 1), len = e1 - e0;
      if (do_sort) {
        if (len <= 128) {  // the row sits in registers (4 entries per lane), ranks by broadcast: no memory round trips
          int c[4];
          float dv[4];
          int rank[4] = {0, 0, 0, 0};
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const int e = lane + 32 * t;
            c[t] = (e < len) ? __ldcg(P.col_tmp + e0 + e) : 0x7fffffff;
            dv[t] = (e < len) ? __ldcg(P.dist_tmp + e0 + e) : 0.f;
          }
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            if (32 * t >= len) break;  // warp-uniform
            const int cnt = min(32, len - 32 * t);
            for (int f = 0; f < cnt; ++f) {
              const int o = __shfl_sync(FULL, c[t], f);
#pragma unroll
              for (int u = 0; u < 4; ++u) rank[u] += (o < c[u]);
            }
          }
#pragma unroll
          for (int t = 0; t < 4; ++t)
            if (lane + 32 * t < len) {
              P.col[e0 + rank[t]] = c[t];
              P.dist[e0 + rank[t]] = dv[t];
            }
        } else {
          for (int e = lane; e < len; e += 32) {
            const int c = __ldcg(P.col_tmp + e0 + e);
            int rank = 0;
            for (int f = 0; f < len; ++f) rank += (__ldcg(P.col_tmp + e0 + f) < c);
            P.col[e0 + rank] = c;
            P.dist[e0 + rank] = __ldcg(P.dist_tmp + e0 + e);
          }
        }
        __syncwarp();  // the row's sorted entries (written by other lanes) are read below
      }
      if (!do_weights) continue;
      const float ei_f = P.eps_auto ? __ldg(P.knn_dist + (size_t)i * k + (k - 1)) : P.eps_fixed;
      if (lane == 0) {
        P.eps[i] = ei_f;
        P.kappa[i] = P.eps_auto ? __ldg(P.knn_idx + (size_t)i * k + (k - 1)) : -1;
        if (ei_f < 1e-10f && P.info != nullptr) atomicOr(&P.info[GLL_INFO_STATUS], GLL_STATUS_EPS_TINY);
      }
      const double ei = (double)ei_f;
      double dsum = 0.0;
      int uu = 0;
      for (int e = e0 + lane; e < e1; e += 32) {
        const int j = P.col[e];
        const double dd = (double)P.dist[e];
        const double ej = P.eps_auto ? (double)__ldg(P.knn_dist + (size_t)j * k + (k - 1)) : (double)P.eps_fixed;
        const float wv = (float)exp(-4.0 * dd * dd / ei / ej);
        P.w[e] = wv;
        dsum += (double)wv;
        uu += (j >= k_lab);
      }
      dsum = warp_sum(dsum);
      uu = warp_sum(uu);
      if (lane == 0) P.deg[i] = (float)dsum;
      if (i < k_lab) {
        // ut[:k_lab] = Y  (GLL.py:109)
        for (int c = lane; c < lp; c += 32) P.ut[(size_t)i * lp + c] = (c < l) ? P.Y[(size_t)i * l + c] : 0.f;
        continue;
      }
      const int r = i - k_lab;
      if (lane == 0) {
        P.uu_cnt[r] = uu;
        P.diag[r] = (float)(dsum + (double)P.tau);
      }
      __syncwarp();  // w of this row, written by other lanes
      // rhs_r = sum over labeled neighbours (sorted columns: they are the head of the row)
      const int e_lab_end = e1 - uu;
      for (int c = lane; c < lp; c += 32) {
        double acc = 0.0;
        if (c < l)
          for (int e = e0; e < e_lab_end; ++e) acc += (double)P.w[e] * (double)__ldg(P.Y + (size_t)P.col[e] * l + c);
        P.rhs[(size_t)r * lp + c] = (float)acc;
      }
    }
    if (P.phase_end > 4) gf_barrier(P.counter, target);
    GF_STAMP(4);
    ++ph;
  }
  // ---- 4: uu_ptr ----
  const int m = n - P.k_lab;
  if (ph == 4 && ph < P.phase_end) {
    grid_scan(P.uu_cnt, m, P.uu_ptr, P.tile_sums, P.counter, target, sm);
    gf_barrier(P.counter, target);
    GF_STAMP(5);
    ++ph;
  }
  // ---- 5: compact off-diagonal CSR of L_uu (columns rebased to the unlabeled block) ----
  if (ph == 5 && ph < P.phase_end) {
    if (gtid == 0 && P.info != nullptr) P.info[GLL_INFO_NNZ_UU] = __ldcg(P.uu_ptr + m);
    for (long long wi = gwarp; wi < m; wi += nwarps) {
      const int r = (int)wi;
      const int o0 = __ldcg(P.uu_ptr + r), cnt = __ldcg(P.uu_ptr + r + 1) - o0;
      const int src = __ldcg(P.row_ptr + P.k_lab + r + 1) - cnt;
      for (int t = lane; t < cnt; t += 32) {
        P.uu_col[o0 + t] = __ldcg(P.col + src + t) - P.k_lab;  // written by other SMs in phase 3: read through L2
        P.uu_val[o0 + t] = __ldcg(P.w + src + t);
      }
    }
  }
  GF_STAMP(6);
#undef GF_STAMP
}

int gf_grid() { return device_info().sms; }
size_t gf_common_bytes() { return 256 + align_up(sizeof(int) * (size_t)(gf_grid() + 1), 256); }

}  // namespace

size_t graph_ws_bytes(int n, int k) {
  size_t emax = gll_max_edges(n, k);
  return align_up(sizeof(int) * (size_t)(n + 1), 256) * 2 + align_up(sizeof(int) * emax, 256) + align_up(sizeof(float) * emax, 256) +
         align_up((size_t)n * k, 256) + gf_common_bytes() + 1024;
}
size_t weights_ws_bytes(int n, int k) {
  (void)k;
  return align_up(sizeof(int) * (size_t)(n + 1), 256) + gf_common_bytes() + 1024;
}
size_t graph_weights_ws_bytes(int n, int k) { return graph_ws_bytes(n, k) + weights_ws_bytes(n, k); }

int graph_stages_run(const GraphBufs& B, const float* Y, int n, int k, int l, int k_lab, int eps_auto, float eps_fixed, float tau,
                     int phase_begin, int phase_end, void* ws, size_t ws_bytes, cudaStream_t st) {
  const bool build = phase_begin == 0;  // K2 from the kNN lists; otherwise the rows are sorted already (col_tmp stays NULL)
  const bool weights = phase_end > 4;   // K3; otherwise phase 3 only sorts the rows (w stays NULL)
  GLL_REQUIRE(B.knn_idx && B.knn_dist && B.row_ptr && B.col && B.dist && ws, "null pointer");
  GLL_REQUIRE(n >= 1 && k >= 2, "bad sizes");
  if (weights) {
    GLL_REQUIRE(B.eps && B.kappa && B.w && B.deg && B.uu_ptr && B.uu_col && B.uu_val && B.diag && B.rhs && B.ut, "null pointer");
    GLL_REQUIRE(k_lab >= 0 && k_lab < n && l >= 1, "need 0 <= k_lab < n and l >= 1");
    GLL_REQUIRE(k_lab == 0 || Y != nullptr, "label matrix missing");
  }
  const size_t need = (build ? graph_ws_bytes(n, k) : 0) + (weights ? weights_ws_bytes(n, k) : 0);
  if (ws_bytes < need) {
    set_error("%s workspace too small: %zu < %zu", build ? "graph" : "weights", ws_bytes, need);
    return GLL_ERR_WORKSPACE;
  }
  GfParams P;
  memset(&P, 0, sizeof(P));
  P.trace = (unsigned long long*)cg_get_trace();
  P.knn_idx = B.knn_idx;
  P.knn_dist = B.knn_dist;
  P.n = n;
  P.k = k;
  P.row_ptr = B.row_ptr;
  P.col = B.col;
  P.dist = B.dist;
  P.info = B.info;
  P.phase_begin = phase_begin;
  P.phase_end = phase_end;
  // common = [barrier counter (256 B) | tile sums], then the K2 scratch, then uu_cnt
  Carver cv(ws, ws_bytes);
  char* common = cv.take<char>(gf_common_bytes());
  P.counter = (unsigned*)common;
  P.tile_sums = (int*)(common + 256);
  size_t zero_bytes = 64;  // the barrier counter
  if (build) {
    const size_t emax = gll_max_edges(n, k);
    P.len = cv.take<int>(n + 1);
    P.cursor = cv.take<int>(n + 1);
    P.col_tmp = cv.take<int>(emax);
    P.dist_tmp = cv.take<float>(emax);
    P.flag = cv.take<unsigned char>((size_t)n * k);
    // the counter, len and cursor are adjacent 256-aligned blocks: ONE memset clears all three
    zero_bytes = (size_t)((char*)P.cursor - common) + sizeof(int) * (size_t)(n + 1);
  }
  if (weights) {
    P.uu_cnt = cv.take<int>(n + 1);
    P.Y = Y;
    P.l = l;
    P.lp = padded_classes(l);
    P.k_lab = k_lab;
    P.eps_auto = eps_auto;
    P.eps_fixed = eps_fixed;
    P.tau = tau;
    P.eps = B.eps;
    P.kappa = B.kappa;
    P.w = B.w;
    P.deg = B.deg;
    P.uu_ptr = B.uu_ptr;
    P.uu_col = B.uu_col;
    P.uu_val = B.uu_val;
    P.diag = B.diag;
    P.rhs = B.rhs;
    P.ut = B.ut;
  }
  GLL_CUDA_CHECK(cudaMemsetAsync(common, 0, zero_bytes, st));
  void* args[] = {&P};
  ProfScope prof(phase_begin == 3 ? KID_WEIGHTS : KID_GRAPH, st);
  GLL_CUDA_CHECK(cudaLaunchCooperativeKernel((const void*)graph_weights_kernel, dim3(gf_grid()), dim3(GF_THREADS), args, 0, st));
  return GLL_OK;
}

}  // namespace gll
