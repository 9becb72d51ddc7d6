// K4 -- persistent multi-right-hand-side Jacobi-CG (replaces spsolve at GLL.py:53 and GLL.py:93; semantics of
// stable_conjgrad GLL.py:247-276: all class columns advance together, per-column freeze once r_c^T r_c <= tol^2,
// stop when max_c ||r_c||_2 <= tol or max_iter; the p = r alias of GLL.py:254 is NOT reproduced).
//
// ONE cooperative launch runs the whole solve.  A = diag - offdiag(val) on the unlabeled block, x0 = 0.
// Per iteration (three grid-wide barriers, the first two carry the dot-product reductions):
//   phase 1  Ap_i = diag_i p_i - sum_j W_ij p_j      warp per row; lane = (neighbour slot s, class quad q): 128-bit
//            gathers of p_j, shuffle reduction over s; fused partial <p, Ap>
//   phase 2  x += a p ; r -= a Ap ; z = r/diag       lanes tile S rows x Q quads = one contiguous 128-bit span per
//            warp; fused partial <r,z>, <r,r>
//   phase 3  p = z + b p
// Reductions are deterministic: per-warp shuffle tree -> per-block fixed-order sum -> per-grid partials
// [column][block] summed by one warp per column in a fixed order (no floating-point atomics anywhere).
// Vectors written by other CTAs are read with ld.global.cg (L2), never through a possibly stale L1 line.
#include <cooperative_groups.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "cg_common.cuh"

namespace gll {
namespace {


__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned& epoch) {
  __syncthreads();
  if (threadIdx.x == 0) {
    epoch += 1;
    __threadfence();
    atomicAdd(counter, 1u);
    const unsigned target = epoch * gridDim.x;
    while (ld_acquire_u32(counter) < target) {
    }
    __threadfence();
  }
  __syncthreads();
}

// Deterministic grid-wide sum of NV float4 accumulators per lane (lane owns class quad q), with a grid barrier.
// out[v*lp + c] (shared, double) holds the result on return.
template <int NV>
__device__ __forceinline__ void grid_reduce(float4 (&acc)[NV], const CgParams& P, int s, int q, int S, int Q, bool active,
                                            double* wpart, double* out, int& buf, unsigned& epoch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lp = P.lp;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    float4 a = active ? acc[v] : make_float4(0.f, 0.f, 0.f, 0.f);
    a = reduce_over_s(a, s, S, Q);
    if (lane < Q) {
      double* d = wpart + ((size_t)v * CG_WARPS + warp) * lp + 4 * lane;
      d[0] = (double)a.x;
      d[1] = (double)a.y;
      d[2] = (double)a.z;
      d[3] = (double)a.w;
    }
  }
  __syncthreads();
  const int G = gridDim.x;
  double* mine = P.partial + (size_t)buf * (2 * CG_MAX_LP) * G;
  for (int c = threadIdx.x; c < NV * lp; c += CG_THREADS) {
    const int v = c / lp, cc = c - v * lp;
    double t = 0.0;
    for (int w = 0; w < CG_WARPS; ++w) t += wpart[((size_t)v * CG_WARPS + w) * lp + cc];
    mine[(size_t)c * G + blockIdx.x] = t;
  }
  grid_barrier(P.barrier, epoch);
  for (int c = warp; c < NV * lp; c += CG_WARPS) {
    double t = 0.0;
    for (int b = lane; b < G; b += 32) t += __ldcg(mine + (size_t)c * G + b);
    t = warp_sum(t);
    if (lane == 0) out[c] = t;
  }
  buf ^= 1;
  __syncthreads();
}

// MASK: the masked operator of laplace_learning_trials.  Column c of this solve is column mask_col0 + c of mask_trials trials
// of mask_cols columns each, and A p is zeroed at (row i, trial t) when mask_slot[i mask_trials + t] >= 0.  MASK = false never
// reads the mask.
template <bool MASK>
__global__ void __launch_bounds__(CG_THREADS, 1) cg_persistent_kernel(CgParams P) {
  extern __shared__ __align__(16) double sm[];
  const int lp = P.lp, Q = lp >> 2, S = 32 / Q;
  double* wpart = sm;                            // [2][CG_WARPS][lp]
  double* red = wpart + 2 * CG_WARPS * lp;       // [2*lp]
  double* rz = red + 2 * lp;                     // [lp]
  double* rr = rz + lp;                          // [lp]
  float* alpha = reinterpret_cast<float*>(rr + lp);  // [lp]
  float* beta = alpha + lp;                          // [lp]

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int s = lane / Q, q = lane - s * Q;
  const bool active = lane < S * Q;
  const int row_begin = blockIdx.x * P.rows_per_block;
  const int row_end = min(P.m, row_begin + P.rows_per_block);
  double tol = (double)P.tol, tol2 = tol * tol;  // P.tol < 0: relative, resolved after the initial reduction
  unsigned epoch = 0;
  int buf = 0;

  // ---- init: x = 0, r = b, p = z = r/diag ----
  {
    float4 acc[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
    for (int i0 = row_begin + warp * S; i0 < row_end; i0 += CG_WARPS * S) {
      const int i = i0 + s;
      if (active && i < row_end) {
        const size_t o = (size_t)i * lp + 4 * q;
        const float4 b = ldcg4(P.rhs + o);
        const float dinv = 1.f / __ldg(P.diag + i);
        const float4 z = make_float4(b.x * dinv, b.y * dinv, b.z * dinv, b.w * dinv);
        st4(P.x + o, make_float4(0.f, 0.f, 0.f, 0.f));
        st4(P.r + o, b);
        st4(P.p + o, z);
        acc[0].x += b.x * z.x; acc[0].y += b.y * z.y; acc[0].z += b.z * z.z; acc[0].w += b.w * z.w;
        acc[1].x += b.x * b.x; acc[1].y += b.y * b.y; acc[1].z += b.z * b.z; acc[1].w += b.w * b.w;
      }
    }
    grid_reduce<2>(acc, P, s, q, S, Q, active, wpart, red, buf, epoch);
    for (int c = threadIdx.x; c < lp; c += CG_THREADS) {
      rz[c] = red[c];
      rr[c] = red[lp + c];
    }
    __syncthreads();
    if (P.tol < 0.f) {  // relative to the largest right-hand-side column norm (every thread computes the same value)
      double mx = 0.0;
      for (int c = 0; c < lp; ++c) mx = fmax(mx, rr[c]);
      tol = -(double)P.tol * sqrt(mx);
      tol2 = tol * tol;
    }
  }

  int it = 0;
  bool nonfinite = false;
  double maxrr = 0.0;
  while (true) {
    maxrr = 0.0;
    for (int c = 0; c < lp; ++c) {
      const double v = rr[c];
      if (!(v == v) || isinf(v)) nonfinite = true;
      maxrr = fmax(maxrr, v);
    }
    if (nonfinite || sqrt(maxrr) <= tol || it >= P.max_iter) break;
    ++it;

    // ---- phase 1: Ap = A p, partial <p, Ap> ----
    float4 dot[1] = {make_float4(0.f, 0.f, 0.f, 0.f)};
    for (int i = row_begin + warp; i < row_end; i += CG_WARPS) {
      const int e0 = __ldg(P.ptr + i), e1 = __ldg(P.ptr + i + 1);
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
      if (active) {
        // four neighbours per trip: the four 128-bit gathers are independent, so a row of ~26 neighbours costs ~7 memory
        // round trips instead of 26 (with many class columns a warp has a single neighbour slot, S = 1)
        for (int e = e0 + s; e < e1; e += 4 * S) {
          float wv[4];
          float4 pj[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const int et = e + t * S;
            const bool ok = et < e1;
            const int j = ok ? __ldg(P.col + et) : 0;
            wv[t] = ok ? __ldg(P.val + et) : 0.f;
            pj[t] = ldcg4(P.p + (size_t)j * lp + 4 * q);
          }
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            a.x = fmaf(wv[t], pj[t].x, a.x);
            a.y = fmaf(wv[t], pj[t].y, a.y);
            a.z = fmaf(wv[t], pj[t].z, a.z);
            a.w = fmaf(wv[t], pj[t].w, a.w);
          }
        }
      }
      a = reduce_over_s(a, s, S, Q);
      if (lane < Q) {
        const size_t o = (size_t)i * lp + 4 * lane;
        const float4 pi = ldcg4(P.p + o);
        const float dg = __ldg(P.diag + i);
        float4 ap = make_float4(fmaf(dg, pi.x, -a.x), fmaf(dg, pi.y, -a.y), fmaf(dg, pi.z, -a.z), fmaf(dg, pi.w, -a.w));
        if constexpr (MASK) {  // row i clamped in this quad's trial: r, p and x stay 0 there (a quad never spans two trials)
          const int t = (P.mask_col0 + 4 * lane) / P.mask_cols;
          if (__ldg(P.mask_slot + (size_t)i * P.mask_trials + t) >= 0) ap = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        st4(P.ap + o, ap);
        dot[0].x = fmaf(pi.x, ap.x, dot[0].x);
        dot[0].y = fmaf(pi.y, ap.y, dot[0].y);
        dot[0].z = fmaf(pi.z, ap.z, dot[0].z);
        dot[0].w = fmaf(pi.w, ap.w, dot[0].w);
      }
    }
    // dot lives on lanes < Q only (s == 0): zero the rest so that the s-reduction is a no-op for them
    if (lane >= Q) dot[0] = make_float4(0.f, 0.f, 0.f, 0.f);
    grid_reduce<1>(dot, P, s, q, S, Q, active, wpart, red, buf, epoch);
    for (int c = threadIdx.x; c < lp; c += CG_THREADS) {
      const bool live = rr[c] > tol2;
      alpha[c] = live ? (float)(rz[c] / red[c]) : 0.f;
    }
    __syncthreads();

    // ---- phase 2: x += alpha p, r -= alpha Ap, partial <r,z>, <r,r> ----
    float4 acc[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
    const float4 al = active ? *reinterpret_cast<const float4*>(alpha + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i0 = row_begin + warp * S; i0 < row_end; i0 += CG_WARPS * S) {
      const int i = i0 + s;
      if (active && i < row_end) {
        const size_t o = (size_t)i * lp + 4 * q;
        float4 x = ldcg4(P.x + o), r = ldcg4(P.r + o);
        const float4 p = ldcg4(P.p + o), ap = ldcg4(P.ap + o);
        const float dinv = 1.f / __ldg(P.diag + i);
        x.x = fmaf(al.x, p.x, x.x); x.y = fmaf(al.y, p.y, x.y); x.z = fmaf(al.z, p.z, x.z); x.w = fmaf(al.w, p.w, x.w);
        r.x = fmaf(-al.x, ap.x, r.x); r.y = fmaf(-al.y, ap.y, r.y); r.z = fmaf(-al.z, ap.z, r.z); r.w = fmaf(-al.w, ap.w, r.w);
        st4(P.x + o, x);
        st4(P.r + o, r);
        acc[0].x += r.x * r.x * dinv; acc[0].y += r.y * r.y * dinv; acc[0].z += r.z * r.z * dinv; acc[0].w += r.w * r.w * dinv;
        acc[1].x += r.x * r.x; acc[1].y += r.y * r.y; acc[1].z += r.z * r.z; acc[1].w += r.w * r.w;
      }
    }
    grid_reduce<2>(acc, P, s, q, S, Q, active, wpart, red, buf, epoch);
    for (int c = threadIdx.x; c < lp; c += CG_THREADS) {
      const double rz_new = red[c], rr_new = red[lp + c];
      beta[c] = (rr_new > tol2 && rz[c] != 0.0) ? (float)(rz_new / rz[c]) : 0.f;
      rz[c] = rz_new;
      rr[c] = rr_new;
    }
    __syncthreads();

    // ---- phase 3: p = z + beta p ----
    const float4 be = active ? *reinterpret_cast<const float4*>(beta + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i0 = row_begin + warp * S; i0 < row_end; i0 += CG_WARPS * S) {
      const int i = i0 + s;
      if (active && i < row_end) {
        const size_t o = (size_t)i * lp + 4 * q;
        const float4 r = ldcg4(P.r + o);
        float4 p = ldcg4(P.p + o);
        const float dinv = 1.f / __ldg(P.diag + i);
        p.x = fmaf(be.x, p.x, r.x * dinv);
        p.y = fmaf(be.y, p.y, r.y * dinv);
        p.z = fmaf(be.z, p.z, r.z * dinv);
        p.w = fmaf(be.w, p.w, r.w * dinv);
        st4(P.p + o, p);
      }
    }
    grid_barrier(P.barrier, epoch);
  }

  if (blockIdx.x == 0 && threadIdx.x == 0) cg_write_stats(P, it, (float)sqrt(maxrr), nonfinite, sqrt(maxrr), tol);
}

size_t cg_smem_bytes(int lp) {
  return sizeof(double) * ((size_t)2 * CG_WARPS * lp + 2 * lp + 2 * lp) + sizeof(float) * 2 * lp;
}

// Streaming kernel: the layer's conversions run as separate kernels around the solve.
int cg_streaming_launch(CgParams P, cudaStream_t st) {
  const int m = P.m, l = P.l, lp = P.lp;
  if (P.rhs_src != nullptr) {
    const int rc = pack_grad(P.rhs_src, P.rhs_kind == 2, m, l, lp, const_cast<float*>(P.rhs), st, nullptr, 0, P.rhs_scale, P.rhs_scale_f64);
    if (rc) return rc;
    P.rhs_src = nullptr;
  }
  void* x_copy = P.x_copy;
  P.x_copy = nullptr;
  const int grid = max(1, min(ceil_div(m, CG_WARPS), device_info().sms));
  const int S = 32 / (lp / 4);
  P.rows_per_block = ceil_div(ceil_div(m, grid), S) * S;  // keep phase-2/3 spans aligned to whole lane groups
  const void* kern = P.mask_slot ? (const void*)cg_persistent_kernel<true> : (const void*)cg_persistent_kernel<false>;
  GLL_CUDA_CHECK(set_max_dynamic_smem_once(kern, (int)cg_smem_bytes(CG_MAX_LP)));
  GLL_CUDA_CHECK(cudaMemsetAsync(P.barrier, 0, 256, st));
  void* args[] = {&P};
  GLL_PROF(KID_CG, st);
  GLL_CUDA_CHECK(cudaLaunchCooperativeKernel(kern, dim3(grid), dim3(CG_THREADS), args, cg_smem_bytes(lp), st));
  return x_copy ? unpack_pred(P.x, m, l, lp, x_copy, P.x_copy_f64, st) : GLL_OK;
}

}  // namespace

// More than CG_MAX_LP class columns (the reference has no limit): the columns of a multi-right-hand-side CG are independent
// (per-column alpha / beta, GLL.py:262-269), so the solve runs in chunks of CG_MAX_LP columns on packed copies.
__global__ void cg_combine_stats_kernel(const int* __restrict__ iters, const float* __restrict__ resid, int chunks, int* iters_out,
                                        float* resid_out) {
  int it = 0;
  float rs = 0.f;
  for (int c = 0; c < chunks; ++c) {
    it = max(it, iters[c]);
    rs = fmaxf(rs, resid[c]);
  }
  if (iters_out) *iters_out = it;
  if (resid_out) *resid_out = rs;
}

size_t cg_ws_bytes(int m, int l) {
  if (padded_classes(l) > CG_MAX_LP)
    return 2 * align_up(sizeof(float) * (size_t)m * CG_MAX_LP, 256) + 2 * 256 * ceil_div(l, CG_MAX_LP) + 1024 + cg_ws_bytes(m, CG_MAX_LP);
  const int lp = padded_classes(l);
  size_t v = align_up(sizeof(float) * (size_t)m * lp, 256);
  return 3 * v + align_up(sizeof(double) * 2 * (2 * CG_MAX_LP) * (size_t)device_info().sms, 256) + 256 + 1024 +
         cg_resident_ws_bytes(m, lp);
}

// Systems that fit on chip (every config except the sharded 1M-node graph) take an on-chip kernel.  The cluster kernel gathers
// neighbour rows through distributed shared memory, which moves few transactions per clock: it wins on SPARSE systems (C2: 1.4
// off-diagonal entries per row, C3: 3.2 -- 35 us per solve against 41 for the one-CTA kernel) and loses on dense ones (C1: 14.5
// per row -- 154 us against 94 for the multi-CTA kernel).  The host cannot see nnz; the layer passes what it expects,
// (k - 1) m / n, and callers that pass nothing get the other kernels.  GLL_B200_CG_PATH ("streaming" / "resident" / "small" /
// "cluster") is a testing knob: "small" and "cluster" put that kernel first, any other value skips both minibatch kernels.
int cg_pick(int m, int lp, float uu_degree_hint, bool masked) {
  if (masked) return GLL_CG_KERNEL_STREAMING;
  const char* force = getenv("GLL_B200_CG_PATH");
  const bool unset = force == nullptr || force[0] == 0;
  const bool small = !unset && strcmp(force, "small") == 0, cluster = !unset && strcmp(force, "cluster") == 0;
  if (!unset && strcmp(force, "streaming") == 0) return GLL_CG_KERNEL_STREAMING;
  if (unset || small || cluster) {
    const bool sparse = uu_degree_hint > 0.f && uu_degree_hint <= 5.f;
    if ((cluster || (unset && sparse)) && cg_cluster_fits(m, lp)) return GLL_CG_KERNEL_CLUSTER;
    if (cg_small_fits(m, lp)) return GLL_CG_KERNEL_SMALL;
  }
  return cg_resident_fits(m, lp) ? GLL_CG_KERNEL_RESIDENT : GLL_CG_KERNEL_STREAMING;
}

int cg_run(const CgSolve& S, void* ws, size_t ws_bytes, cudaStream_t st) {
  GLL_REQUIRE(S.ptr && S.col && S.val && S.diag && S.rhs && S.x && ws, "null pointer");
  const int m = S.m, l = S.l, lp = padded_classes(l);
  if (ws_bytes < cg_ws_bytes(m, l)) {
    set_error("CG workspace too small: %zu < %zu", ws_bytes, cg_ws_bytes(m, l));
    return GLL_ERR_WORKSPACE;
  }
  Carver cv(ws, ws_bytes);
  if (lp > CG_MAX_LP) {
    if (S.rhs_src != nullptr) {
      const int rc = pack_grad(S.rhs_src, S.rhs_kind == 2, m, l, lp, const_cast<float*>(S.rhs), st, nullptr, 0, S.rhs_scale, S.rhs_scale_f64);
      if (rc) return rc;
    }
    const int chunks = ceil_div(l, CG_MAX_LP);
    float* rhs_c = cv.take<float>((size_t)m * CG_MAX_LP);
    float* x_c = cv.take<float>((size_t)m * CG_MAX_LP);
    int* it_c = cv.take<int>(chunks);
    float* rs_c = cv.take<float>(chunks);
    const size_t sub_bytes = cg_ws_bytes(m, CG_MAX_LP);
    void* sub = cv.take<char>(sub_bytes);
    GLL_CUDA_CHECK(cudaMemsetAsync(S.x, 0, sizeof(float) * (size_t)m * lp, st));  // padded class columns read as zero
    for (int c = 0; c < chunks; ++c) {
      const int c0 = c * CG_MAX_LP, cnt = min(CG_MAX_LP, l - c0), lpc = padded_classes(cnt);
      int rc = pack_columns(S.rhs, m, lp, c0, cnt, rhs_c, lpc, st);
      if (rc) return rc;
      // a chunk: packed columns, no conversions, no sparsity hint; the mask is indexed by the chunk's global columns
      CgSolve C = S;
      C.rhs = rhs_c;
      C.x = x_c;
      C.l = cnt;
      C.iters_out = it_c + c;
      C.resid_out = rs_c + c;
      C.rhs_src = nullptr;
      C.rhs_scale = nullptr;
      C.x_copy = nullptr;
      C.uu_degree_hint = 0.f;
      C.mask_col0 = S.mask_col0 + c0;
      rc = cg_run(C, sub, sub_bytes, st);
      if (rc) return rc;
      rc = unpack_columns(x_c, m, lpc, c0, cnt, S.x, lp, st);
      if (rc) return rc;
    }
    cg_combine_stats_kernel<<<1, 1, 0, st>>>(it_c, rs_c, chunks, S.iters_out, S.resid_out);
    GLL_LAUNCH_CHECK();
    return S.x_copy ? unpack_pred(S.x, m, l, lp, S.x_copy, S.x_copy_f64, st) : GLL_OK;
  }
  CgParams P{S};
  P.lp = lp;
  P.r = cv.take<float>((size_t)m * lp);
  P.p = cv.take<float>((size_t)m * lp);
  P.ap = cv.take<float>((size_t)m * lp);
  P.partial = cv.take<double>((size_t)2 * (2 * CG_MAX_LP) * device_info().sms);
  P.barrier = cv.take<unsigned>(64);
  void* scratch = cv.take<char>(cg_resident_ws_bytes(m, lp));
  switch (cg_pick(m, lp, S.uu_degree_hint, S.mask_slot != nullptr)) {
    case GLL_CG_KERNEL_CLUSTER: return cg_cluster_launch(P, st);    // one cluster of eight CTAs (64 <= m <= 2048)
    case GLL_CG_KERNEL_SMALL: return cg_small_launch(P, st);        // one CTA (m <= 512)
    case GLL_CG_KERNEL_RESIDENT: return cg_resident_launch(P, scratch, st);
    default: return cg_streaming_launch(P, st);
  }
}

}  // namespace gll
