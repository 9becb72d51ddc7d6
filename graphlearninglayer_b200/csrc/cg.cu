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


__device__ __forceinline__ unsigned ld_acquire(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned& epoch) {
  __syncthreads();
  if (threadIdx.x == 0) {
    epoch += 1;
    __threadfence();
    atomicAdd(counter, 1u);
    const unsigned target = epoch * gridDim.x;
    while (ld_acquire(counter) < target) {
    }
    __threadfence();
  }
  __syncthreads();
}

__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// sum over the neighbour-slot index s of lane = s*Q + q; result valid on lanes < Q
__device__ __forceinline__ float4 reduce_over_s(float4 a, int s, int S, int Q) {
  int top = 1;
  while (top < S) top <<= 1;
  int span = S;
  for (int st = top >> 1; st >= 1; st >>= 1) {
    float4 o;
    o.x = __shfl_down_sync(FULL, a.x, st * Q);
    o.y = __shfl_down_sync(FULL, a.y, st * Q);
    o.z = __shfl_down_sync(FULL, a.z, st * Q);
    o.w = __shfl_down_sync(FULL, a.w, st * Q);
    if (s < st && s + st < span) {
      a.x += o.x;
      a.y += o.y;
      a.z += o.z;
      a.w += o.w;
    }
    span = min(span, st);
  }
  return a;
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

// Masked operator of laplace_learning_trials: column c of this solve is column col0 + c of `trials` trials of `cols` columns each,
// and A p is zeroed at (row i, trial t) when slot[i trials + t] >= 0.  A separate parameter, so that CgParams (shared with the
// on-chip kernels) keeps its layout.
struct CgMask {
  const int* slot;
  int trials, cols, col0;
};

// MASK = false is the unmasked solve and never reads M
template <bool MASK>
__global__ void __launch_bounds__(CG_THREADS, 1) cg_persistent_kernel(CgParams P, CgMask M) {
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
          const int t = (M.col0 + 4 * lane) / M.cols;
          if (__ldg(M.slot + (size_t)i * M.trials + t) >= 0) ap = make_float4(0.f, 0.f, 0.f, 0.f);
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

  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const float resid = (float)sqrt(maxrr);
    if (P.iters_out) *P.iters_out = it;
    if (P.resid_out) *P.resid_out = resid;
    if (P.status_out) {
      int st = 0;
      if (nonfinite) st |= GLL_STATUS_NONFINITE;
      if (!nonfinite && !(sqrt(maxrr) <= tol)) st |= GLL_STATUS_CG_NOT_CONVERGED;
      if (st) atomicOr(P.status_out, st);
    }
  }
}

size_t cg_smem_bytes(int lp) {
  return sizeof(double) * ((size_t)2 * CG_WARPS * lp + 2 * lp + 2 * lp) + sizeof(float) * 2 * lp;
}

int cg_grid(int m) {
  int g = ceil_div(m, CG_WARPS);
  return max(1, min(g, device_info().sms));
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

int cg_run(const int* uu_ptr, const int* uu_col, const float* uu_val, const float* diag, const float* rhs, int m, int l,
           float tol, int max_iter, float* x, int* iters_out, float* resid_out, int* status_out, void* ws, size_t ws_bytes,
           cudaStream_t st, unsigned* ext_counter, const CgIo* io) {
  GLL_REQUIRE(uu_ptr && uu_col && uu_val && diag && rhs && x && ws, "null pointer");
  const int lp = padded_classes(l);
  if (ws_bytes < cg_ws_bytes(m, l)) {
    set_error("CG workspace too small: %zu < %zu", ws_bytes, cg_ws_bytes(m, l));
    return GLL_ERR_WORKSPACE;
  }
  Carver cv(ws, ws_bytes);
  // Layer-side conversions (GLL.py:66 float64 output, GLL.py:104 the incoming gradient): the on-chip kernels read / write the
  // caller's arrays themselves; the chunked and the streaming path run the two small kernels around the solve.
  const bool has_src = io != nullptr && io->rhs_src != nullptr, has_copy = io != nullptr && io->x_copy != nullptr;
  const bool masked = io != nullptr && io->mask_slot != nullptr;
  if (lp > CG_MAX_LP) {
    if (has_src) {
      const int rc = pack_grad(io->rhs_src, io->rhs_kind == 2, m, l, lp, const_cast<float*>(rhs), st, nullptr, 0, io->rhs_scale, io->rhs_scale_f64);
      if (rc) return rc;
    }
    const int chunks = ceil_div(l, CG_MAX_LP);
    float* rhs_c = cv.take<float>((size_t)m * CG_MAX_LP);
    float* x_c = cv.take<float>((size_t)m * CG_MAX_LP);
    int* it_c = cv.take<int>(chunks);
    float* rs_c = cv.take<float>(chunks);
    const size_t sub_bytes = cg_ws_bytes(m, CG_MAX_LP);
    void* sub = cv.take<char>(sub_bytes);
    GLL_CUDA_CHECK(cudaMemsetAsync(x, 0, sizeof(float) * (size_t)m * lp, st));  // padded class columns read as zero
    for (int c = 0; c < chunks; ++c) {
      const int c0 = c * CG_MAX_LP, cnt = min(CG_MAX_LP, l - c0), lpc = padded_classes(cnt);
      int rc = pack_columns(rhs, m, lp, c0, cnt, rhs_c, lpc, st);
      if (rc) return rc;
      CgIo mio = {};  // a masked solve: the mask is indexed by the chunk's global columns
      if (masked) {
        mio.mask_slot = io->mask_slot;
        mio.mask_trials = io->mask_trials;
        mio.mask_cols = io->mask_cols;
        mio.mask_col0 = io->mask_col0 + c0;
      }
      rc = cg_run(uu_ptr, uu_col, uu_val, diag, rhs_c, m, cnt, tol, max_iter, x_c, it_c + c, rs_c + c, status_out, sub, sub_bytes, st,
                  ext_counter, masked ? &mio : nullptr);
      if (rc) return rc;
      rc = unpack_columns(x_c, m, lpc, c0, cnt, x, lp, st);
      if (rc) return rc;
    }
    cg_combine_stats_kernel<<<1, 1, 0, st>>>(it_c, rs_c, chunks, iters_out, resid_out);
    GLL_LAUNCH_CHECK();
    return has_copy ? unpack_pred(x, m, l, lp, io->x_copy, io->x_copy_f64, st) : GLL_OK;
  }
  CgParams P;
  P.ptr = uu_ptr;
  P.col = uu_col;
  P.val = uu_val;
  P.diag = diag;
  P.rhs = rhs;
  P.x = x;
  P.r = cv.take<float>((size_t)m * lp);
  P.p = cv.take<float>((size_t)m * lp);
  P.ap = cv.take<float>((size_t)m * lp);
  P.partial = cv.take<double>((size_t)2 * (2 * CG_MAX_LP) * device_info().sms);
  P.barrier = cv.take<unsigned>(64);
  P.m = m;
  P.l = l;
  P.lp = lp;
  P.max_iter = max_iter;
  P.tol = tol;
  P.iters_out = iters_out;
  P.resid_out = resid_out;
  P.status_out = status_out;
  P.rows_per_block = 0;
  P.ext_counter = ext_counter;
  P.rhs_src = io ? io->rhs_src : nullptr;
  P.rhs_kind = io ? io->rhs_kind : 0;
  P.x_copy = io ? io->x_copy : nullptr;
  P.x_copy_f64 = io ? io->x_copy_f64 : 0;
  P.rhs_scale = io ? io->rhs_scale : nullptr;
  P.rhs_scale_f64 = io ? io->rhs_scale_f64 : 0;
  if (!masked) {  // systems that fit on chip (every config except the sharded 1M-node graph) take the shared-memory-resident kernel
    const char* force = getenv("GLL_B200_CG_PATH");  // "streaming" / "resident" / "small" / "cluster": testing knobs
    const bool only_small = force != nullptr && strcmp(force, "small") == 0;
    const bool force_cluster = force != nullptr && strcmp(force, "cluster") == 0;
    // The cluster kernel gathers neighbour rows through distributed shared memory, which moves few transactions per clock: it
    // wins on SPARSE systems (C2: 1.4 off-diagonal entries per row, C3: 3.2 -- 35 us per solve against 41 for the one-CTA kernel)
    // and loses on dense ones (C1: 14.5 per row -- 154 us against 94 for the multi-CTA kernel).  The host cannot see nnz; the
    // layer passes what it expects, (k - 1) m / n, and callers that pass nothing get the other kernels.
    const bool sparse = io != nullptr && io->uu_degree_hint > 0.f && io->uu_degree_hint <= 5.f;
    if (force == nullptr || force[0] == 0 || only_small || force_cluster) {  // minibatch-sized systems: the latency-organised kernels
      int rc = (force_cluster || (sparse && !only_small)) ? cg_cluster_try(P, st) : 0;  // one cluster of eight CTAs (64 <= m <= 2048)
      if (rc < 0) return rc;
      if (rc == 1) return GLL_OK;
      rc = cg_small_try(P, st);  // one CTA, a thread per row (m <= 512)
      if (rc < 0) return rc;
      if (rc == 1) return GLL_OK;
    }
    if (!(force && strcmp(force, "streaming") == 0)) {
      void* scratch = cv.take<char>(cg_resident_ws_bytes(m, lp));
      const int rc = cg_resident_try(P, scratch, st);
      if (rc < 0) return rc;
      if (rc == 1) return GLL_OK;
    }
  }
  if (has_src) {  // streaming kernel: conversions as separate kernels
    const int rc = pack_grad(io->rhs_src, io->rhs_kind == 2, m, l, lp, const_cast<float*>(rhs), st, nullptr, 0, io->rhs_scale, io->rhs_scale_f64);
    if (rc) return rc;
    P.rhs_src = nullptr;
  }
  P.x_copy = nullptr;
  const int grid = cg_grid(m);
  const int S = 32 / (lp / 4);
  int rpb = ceil_div(m, grid);
  rpb = ceil_div(rpb, S) * S;  // keep phase-2/3 spans aligned to whole lane groups
  P.rows_per_block = rpb;
  const size_t smem = cg_smem_bytes(lp);
  const void* kern = masked ? (const void*)cg_persistent_kernel<true> : (const void*)cg_persistent_kernel<false>;
  GLL_CUDA_CHECK(set_max_dynamic_smem_once(kern, (int)cg_smem_bytes(CG_MAX_LP)));
  GLL_CUDA_CHECK(cudaMemsetAsync(P.barrier, 0, 256, st));
  CgMask M = {nullptr, 0, 0, 0};
  if (masked) M = {io->mask_slot, io->mask_trials, io->mask_cols, io->mask_col0};
  void* args[] = {&P, &M};
  GLL_PROF(KID_CG, st);
  GLL_CUDA_CHECK(cudaLaunchCooperativeKernel(kern, dim3(grid), dim3(CG_THREADS), args, smem, st));
  return has_copy ? unpack_pred(x, m, l, lp, io->x_copy, io->x_copy_f64, st) : GLL_OK;
}

}  // namespace gll
