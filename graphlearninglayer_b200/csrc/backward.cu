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

constexpr int ROW_CHUNK = 128;

template <int W>
__device__ __forceinline__ void load_chunk(const float* __restrict__ base, int c, float (&v)[W]) {
  if constexpr (W == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(base) + c);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
    v[0] = __ldg(base + c);
  }
}

// block per row; a thread owns up to 4 feature chunks (W floats each) per pass and keeps them in registers
template <int W>
__global__ void __launch_bounds__(256)
row_gather_kernel(const float* __restrict__ X, int row_begin, int d, int eps_auto, const int* __restrict__ row_ptr,
                  const int* __restrict__ col, const int* __restrict__ kappa, const float* __restrict__ gv,
                  const float* __restrict__ bvec, float* __restrict__ dX) {
  __shared__ int sj[ROW_CHUNK];
  __shared__ float stc[ROW_CHUNK];
  const int i = row_begin + blockIdx.x;
  const int e0 = row_ptr[i], e1 = row_ptr[i + 1];
  const int ki = eps_auto ? kappa[i] : -1;
  const float bi = eps_auto ? bvec[i] : 0.f;
  const int cols = d / W;
  const float* xrow = X + (size_t)i * d;
  for (int cbase = 0; cbase < cols; cbase += 4 * blockDim.x) {
    double acc[4][W];
    float xi[4][W];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = cbase + u * blockDim.x + threadIdx.x;
#pragma unroll
      for (int t = 0; t < W; ++t) acc[u][t] = 0.0, xi[u][t] = 0.f;
      if (c < cols) load_chunk<W>(xrow, c, xi[u]);
    }
    for (int eb = e0; eb < e1; eb += ROW_CHUNK) {
      const int cnt = min(ROW_CHUNK, e1 - eb);
      __syncthreads();
      for (int t = threadIdx.x; t < cnt; t += blockDim.x) {
        const int j = col[eb + t];
        float tc = gv[eb + t];
        if (eps_auto) {
          if (j == ki) tc -= bi;
          if (kappa[j] == i) tc -= bvec[j];
        }
        sj[t] = j;
        stc[t] = tc;
      }
      __syncthreads();
      for (int t = 0; t < cnt; ++t) {
        const float tc = stc[t];
        if (tc == 0.f) continue;
        const float* xj = X + (size_t)sj[t] * d;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int c = cbase + u * blockDim.x + threadIdx.x;
          if (c < cols) {
            float v[W];
            load_chunk<W>(xj, c, v);
#pragma unroll
            for (int q = 0; q < W; ++q) acc[u][q] += (double)tc * ((double)xi[u][q] - (double)v[q]);
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = cbase + u * blockDim.x + threadIdx.x;
      if (c < cols) {
        if constexpr (W == 4) {
          reinterpret_cast<float4*>(dX + (size_t)i * d)[c] =
              make_float4((float)acc[u][0], (float)acc[u][1], (float)acc[u][2], (float)acc[u][3]);
        } else {
          dX[(size_t)i * d + c] = (float)acc[u][0];
        }
      }
    }
  }
}

// Warp per row (vectorised path, d % 4 == 0): a lane owns NV float4 chunks of the feature row (chunk = lane + 32 u), so one
// neighbour row is NV coalesced 512-byte loads.  Edge metadata (column, t_ij) is prepared 32 edges at a time, one edge per
// lane; edges with t_ij == 0 (both ends labeled: most edges of a minibatch graph) are dropped with a ballot; the row of
// the NEXT surviving edge is already in flight while the current one is accumulated (fp64 accumulators).
// Four rows per CTA: many more rows in flight per SM than the block-per-row kernel, whose CTAs spent their life waiting on
// five dependent loads.
template <int NV>
__global__ void __launch_bounds__(128)
row_gather_warp_kernel(const float* __restrict__ X, int row_begin, int row_end, int d, int eps_auto, const int* __restrict__ row_ptr,
                       const int* __restrict__ col, const int* __restrict__ kappa, const float* __restrict__ gv,
                       const float* __restrict__ bvec, float* __restrict__ dX) {
  const int lane = threadIdx.x & 31;
  // rows are taken from the END: an unlabeled row (they come last, GLL.py:11) gathers ~30 neighbour rows one after the other,
  // a labeled row one or two -- started last, the long chains were the kernel's tail (35 us at C2 for 60 MB of gathers)
  const int i = row_end - 1 - (blockIdx.x * 4 + (threadIdx.x >> 5));
  if (i < row_begin) return;
  const int cols = d >> 2;
  const int e0 = __ldg(row_ptr + i), e1 = __ldg(row_ptr + i + 1);
  const int ki = eps_auto ? __ldg(kappa + i) : -1;
  const float bi = eps_auto ? __ldg(bvec + i) : 0.f;
  const float4* xrow = reinterpret_cast<const float4*>(X + (size_t)i * d);
  for (int cbase = 0; cbase < cols; cbase += 32 * NV) {
    float4 xi[NV];
    double acc[NV][4];
#pragma unroll
    for (int u = 0; u < NV; ++u) {
      const int c = cbase + lane + 32 * u;
      xi[u] = (c < cols) ? __ldg(xrow + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      acc[u][0] = acc[u][1] = acc[u][2] = acc[u][3] = 0.0;
    }
    auto fetch = [&](int j, float4 (&v)[NV]) {
      const float4* xj = reinterpret_cast<const float4*>(X + (size_t)j * d);
#pragma unroll
      for (int u = 0; u < NV; ++u) {
        const int c = cbase + lane + 32 * u;
        v[u] = (c < cols) ? __ldg(xj + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    auto accumulate = [&](float tc, const float4 (&v)[NV]) {
      const double t = (double)tc;
#pragma unroll
      for (int u = 0; u < NV; ++u) {  // the difference is exact enough in fp32 (one rounding); products and sums in fp64
        acc[u][0] = fma(t, (double)(xi[u].x - v[u].x), acc[u][0]);
        acc[u][1] = fma(t, (double)(xi[u].y - v[u].y), acc[u][1]);
        acc[u][2] = fma(t, (double)(xi[u].z - v[u].z), acc[u][2]);
        acc[u][3] = fma(t, (double)(xi[u].w - v[u].w), acc[u][3]);
      }
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
      float4 va[NV], vb[NV];
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
    float4* out = reinterpret_cast<float4*>(dX + (size_t)i * d);
#pragma unroll
    for (int u = 0; u < NV; ++u) {
      const int c = cbase + lane + 32 * u;
      if (c < cols) out[c] = make_float4((float)acc[u][0], (float)acc[u][1], (float)acc[u][2], (float)acc[u][3]);
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
    int threads = min(256, max(32, ceil_div(cols, 32) * 32));
    GLL_PROF(KID_ROW_GATHER, st);
    if (vec4) {
      const int grid = ceil_div(rows, 4);
      if (cols <= 32)
        row_gather_warp_kernel<1><<<grid, 128, 0, st>>>(X, row_begin, row_end, d, eps_auto, B.row_ptr, B.col, B.kappa, B.gv, B.bvec, dX);
      else if (cols <= 64)
        row_gather_warp_kernel<2><<<grid, 128, 0, st>>>(X, row_begin, row_end, d, eps_auto, B.row_ptr, B.col, B.kappa, B.gv, B.bvec, dX);
      else
        row_gather_warp_kernel<4><<<grid, 128, 0, st>>>(X, row_begin, row_end, d, eps_auto, B.row_ptr, B.col, B.kappa, B.gv, B.bvec, dX);
    } else
      row_gather_kernel<1><<<rows, threads, 0, st>>>(X, row_begin, d, eps_auto, B.row_ptr, B.col, B.kappa, B.gv, B.bvec, dX);
  }
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

}  // namespace gll
