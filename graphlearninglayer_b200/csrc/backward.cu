// K5 + K6 -- backward edge pass (GLL.py:104-159).
//   K5  G_ij = -<wt_i - wt_j, ut_i - ut_j>   (GLL.py:111-120, the per-class graph.gradient loop collapsed per edge)
//       gv_ij = G_ij V_ij,  V_ij = -8 W_ij/(eps_i eps_j)                                   (GLL.py:146, 217)
//       b_i = sum_j G_ij modV_ij,  modV_ij = d^2 V_ij / (2 eps_i^2)   (auto only)          (GLL.py:126, 218)
//   K6  dX_i = sum_j t_ij (x_i - x_j),  t_ij = gv_ij - [j == kappa(i)] b_i - [kappa(j) == i] b_j
//       == laplacian(G.*V) X - laplacian(C.*b, symmetrized) X                              (GLL.py:128-159)
// K6 is a row-local gather (t is symmetric), so nothing is scattered and no floating-point atomics are used.
#include "common.cuh"

namespace gll {
namespace {

__global__ void __launch_bounds__(256)
edge_grad_kernel(int row_begin, int row_end, int lp, int k_lab, int eps_auto, const int* __restrict__ row_ptr, const int* __restrict__ col,
                 const float* __restrict__ dist, const float* __restrict__ w, const float* __restrict__ eps,
                 const float* __restrict__ ut, const float* __restrict__ wt, float* __restrict__ gv,
                 float* __restrict__ bvec) {
  // rows are taken from the END: the unlabeled rows come last (GLL.py:11) and are the only ones whose edges all carry work, so
  // they start first instead of forming the kernel's tail
  const int i = row_end - 1 - (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (i < row_begin) return;
  const int e0 = row_ptr[i], e1 = row_ptr[i + 1];
  const double ei = (double)eps[i];
  const float4* ui = reinterpret_cast<const float4*>(ut + (size_t)i * lp);
  const float4* wi = reinterpret_cast<const float4*>(wt + (size_t)i * lp);
  const int Q = lp >> 2;
  double bsum = 0.0;
  for (int e = e0 + lane; e < e1; e += 32) {
    const int j = col[e];
    double G = 0.0;
    if (i >= k_lab || j >= k_lab) {  // both labeled: wt_i = wt_j = 0, G = 0
      const float4* uj = reinterpret_cast<const float4*>(ut + (size_t)j * lp);
      const float4* wj = reinterpret_cast<const float4*>(wt + (size_t)j * lp);
      for (int c = 0; c < Q; ++c) {
        // the adjoint solution of a labeled row is zero by definition (GLL.py:104): never read from wt
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 a = (i >= k_lab) ? __ldg(wi + c) : z4, b = (j >= k_lab) ? __ldg(wj + c) : z4, u = __ldg(ui + c), v = __ldg(uj + c);
        G -= ((double)a.x - (double)b.x) * ((double)u.x - (double)v.x);
        G -= ((double)a.y - (double)b.y) * ((double)u.y - (double)v.y);
        G -= ((double)a.z - (double)b.z) * ((double)u.z - (double)v.z);
        G -= ((double)a.w - (double)b.w) * ((double)u.w - (double)v.w);
      }
    }
    const double ej = (double)eps[j];
    const double V = -8.0 * (double)w[e] / ei / ej;
    gv[e] = (float)(G * V);
    if (eps_auto) {
      const double dd = (double)dist[e];
      bsum += G * (dd * dd * V / (ei * ei) / 2.0);
    }
  }
  if (eps_auto) {
    bsum = warp_sum(bsum);
    if (lane == 0) bvec[i] = (float)bsum;
  }
}

// One W-float chunk of a feature row (W = 4: a float4, W = 1: a float), its update acc += t (x_i - x_j) in fp64 accumulators,
// and its store.  float4 chunks take the difference in fp32 (exact enough: one rounding), single floats in fp64; each form
// keeps the results its path has always given.
__device__ __forceinline__ void accumulate_chunk(double (&acc)[4], double t, float4 xi, float4 xj) {
  acc[0] = fma(t, (double)(xi.x - xj.x), acc[0]);
  acc[1] = fma(t, (double)(xi.y - xj.y), acc[1]);
  acc[2] = fma(t, (double)(xi.z - xj.z), acc[2]);
  acc[3] = fma(t, (double)(xi.w - xj.w), acc[3]);
}
__device__ __forceinline__ void accumulate_chunk(double (&acc)[1], double t, float xi, float xj) {
  acc[0] += t * ((double)xi - (double)xj);
}
__device__ __forceinline__ float4 round_chunk(const double (&acc)[4]) {
  return make_float4((float)acc[0], (float)acc[1], (float)acc[2], (float)acc[3]);
}
__device__ __forceinline__ float round_chunk(const double (&acc)[1]) { return (float)acc[0]; }

template <int W> struct Chunk { using T = float; };
template <> struct Chunk<4> { using T = float4; };

// Warp per row: a lane owns NV W-float chunks of the feature row (chunk = lane + 32 u), so one neighbour row is NV coalesced
// loads of 32 W floats.  W = 4 needs d % 4 == 0 and 16-byte aligned X and dX; W = 1 takes any d and alignment.  Edge
// metadata (column, t_ij) is prepared 32 edges at a time, one edge per lane; edges with t_ij == 0 (both ends labeled: most
// edges of a minibatch graph) are dropped with a ballot; the row of the NEXT surviving edge is already in flight while the
// current one is accumulated (fp64 accumulators).  Four rows per CTA: many rows in flight per SM, where a CTA per row spent
// its life waiting on five dependent loads.
template <int W, int NV>
__global__ void __launch_bounds__(128)
row_gather_kernel(const float* __restrict__ X, int row_begin, int row_end, int d, int eps_auto, const int* __restrict__ row_ptr,
                  const int* __restrict__ col, const int* __restrict__ kappa, const float* __restrict__ gv,
                  const float* __restrict__ bvec, float* __restrict__ dX) {
  using V = typename Chunk<W>::T;
  const int lane = threadIdx.x & 31;
  // rows are taken from the END: an unlabeled row (they come last, GLL.py:11) gathers ~30 neighbour rows one after the other,
  // a labeled row one or two -- started last, the long chains were the kernel's tail (35 us at C2 for 60 MB of gathers)
  const int i = row_end - 1 - (blockIdx.x * 4 + (threadIdx.x >> 5));
  if (i < row_begin) return;
  const int cols = W == 4 ? d >> 2 : d;
  const int e0 = __ldg(row_ptr + i), e1 = __ldg(row_ptr + i + 1);
  const int ki = eps_auto ? __ldg(kappa + i) : -1;
  const float bi = eps_auto ? __ldg(bvec + i) : 0.f;
  const V* xrow = reinterpret_cast<const V*>(X + (size_t)i * d);
  for (int cbase = 0; cbase < cols; cbase += 32 * NV) {
    V xi[NV];
    double acc[NV][W];
#pragma unroll
    for (int u = 0; u < NV; ++u) {
      const int c = cbase + lane + 32 * u;
      xi[u] = (c < cols) ? __ldg(xrow + c) : V{};
#pragma unroll
      for (int q = 0; q < W; ++q) acc[u][q] = 0.0;
    }
    auto fetch = [&](int j, V (&v)[NV]) {
      const V* xj = reinterpret_cast<const V*>(X + (size_t)j * d);
#pragma unroll
      for (int u = 0; u < NV; ++u) {
        const int c = cbase + lane + 32 * u;
        v[u] = (c < cols) ? __ldg(xj + c) : V{};
      }
    };
    auto accumulate = [&](float tc, const V (&v)[NV]) {
      const double t = (double)tc;
#pragma unroll
      for (int u = 0; u < NV; ++u) accumulate_chunk(acc[u], t, xi[u], v[u]);
    };
    for (int eb = e0; eb < e1; eb += 32) {
      const int e = eb + lane;
      int j = 0;
      float tc = 0.f;
      if (e < e1) {
        j = __ldg(col + e);
        tc = __ldg(gv + e);
        if (eps_auto) {
          if (j == ki) tc -= bi;
          if (__ldg(kappa + j) == i) tc -= __ldg(bvec + j);
        }
      }
      unsigned live = __ballot_sync(FULL, tc != 0.f);
      if (live == 0) continue;
      V va[NV], vb[NV];
      int t = __ffs(live) - 1;
      live &= live - 1;
      fetch(__shfl_sync(FULL, j, t), va);
      while (true) {
        const float tca = __shfl_sync(FULL, tc, t);
        if (live == 0) {
          accumulate(tca, va);
          break;
        }
        t = __ffs(live) - 1;
        live &= live - 1;
        fetch(__shfl_sync(FULL, j, t), vb);
        accumulate(tca, va);
        const float tcb = __shfl_sync(FULL, tc, t);
        if (live == 0) {
          accumulate(tcb, vb);
          break;
        }
        t = __ffs(live) - 1;
        live &= live - 1;
        fetch(__shfl_sync(FULL, j, t), va);
        accumulate(tcb, vb);
      }
    }
    V* out = reinterpret_cast<V*>(dX + (size_t)i * d);
#pragma unroll
    for (int u = 0; u < NV; ++u) {
      const int c = cbase + lane + 32 * u;
      if (c < cols) out[c] = round_chunk(acc[u]);
    }
  }
}

}  // namespace

int backward_edges_run(const float* X, int n, int d, int l, int k_lab, int eps_auto, const GraphBufs& B, float* dX, int row_begin,
                       int row_end, int phases, cudaStream_t st) {
  GLL_REQUIRE(X && B.row_ptr && B.col && B.dist && B.w && B.eps && B.ut && B.wt && B.gv && B.bvec && dX, "null pointer");
  GLL_REQUIRE(!eps_auto || B.kappa, "kappa missing");
  GLL_REQUIRE(0 <= row_begin && row_begin <= row_end && row_end <= n, "bad row range");
  const int rows = row_end - row_begin;
  if (rows == 0) return GLL_OK;
  const int lp = padded_classes(l);
  if (phases & 1) {  // K5: gv for the rows' edges, b for the rows
    GLL_PROF(KID_EDGE_GRAD, st);
    edge_grad_kernel<<<ceil_div((long long)rows * 32, 256), 256, 0, st>>>(row_begin, row_end, lp, k_lab, eps_auto, B.row_ptr, B.col,
                                                                          B.dist, B.w, B.eps, B.ut, B.wt, B.gv, B.bvec);
  }
  GLL_LAUNCH_CHECK();
  if (phases & 2) {  // K6: needs b of ALL rows (neighbours j with kappa(j) = i)
    const bool vec4 = (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && ((reinterpret_cast<uintptr_t>(dX) & 15) == 0);
    const int cols = vec4 ? d / 4 : d;
    // NV: as few column passes as the registers allow, with few idle lanes (W = 1, NV = 16: 132 registers, no spills).
    // Measured at C2 on a B200 at 1000 W (tools/row_gather_bench.py): d = 130 takes 20.6 us at NV = 8, 28.7 at 16; d = 2051
    // takes 174 us at NV = 16, 218 at 8.
    auto* kernel = vec4 ? (cols <= 32 ? row_gather_kernel<4, 1> : cols <= 64 ? row_gather_kernel<4, 2> : row_gather_kernel<4, 4>)
                        : (cols <= 32    ? row_gather_kernel<1, 1>
                           : cols <= 128 ? row_gather_kernel<1, 4>
                           : cols <= 256 ? row_gather_kernel<1, 8>
                                         : row_gather_kernel<1, 16>);
    GLL_PROF(KID_ROW_GATHER, st);
    kernel<<<ceil_div(rows, 4), 128, 0, st>>>(X, row_begin, row_end, d, eps_auto, B.row_ptr, B.col, B.kappa, B.gv, B.bvec, dX);
  }
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

}  // namespace gll
