// Shared by the CG kernels: cg.cu (streaming: vectors in global memory, any size), the on-chip kernels cg_resident.cu,
// cg_small.cu and cg_cluster.cu, and the row-partitioned cg_rows.cu.
#pragma once
#include "common.cuh"

namespace gll {

constexpr int CG_THREADS = 1024;
constexpr int CG_WARPS = CG_THREADS / 32;
constexpr int CG_MAX_LP = 128;

// The request plus what cg_run derives for the kernels.
// (The field order of CgSolve and CgParams matters to speed: the compiler pairs adjacent parameters in its constant loads, and
// this order gives the streaming kernels the schedule they were tuned with.)
struct CgParams : CgSolve {
  // streaming kernel only
  float* r;
  float* p;
  float* ap;
  double* partial;    // [2 buffers][2*lp columns][grid]
  unsigned* barrier;  // zeroed before launch
  int lp;
  int rows_per_block;
};

__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 scale4(const float4& a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }
__device__ __forceinline__ void fma4(float4& acc, float w, const float4& v) {
  acc.x = fmaf(w, v.x, acc.x);
  acc.y = fmaf(w, v.y, acc.y);
  acc.z = fmaf(w, v.z, acc.z);
  acc.w = fmaf(w, v.w, acc.w);
}
__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

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

// Chronopoulos-Gear vector update of one class quad (every kernel but the streaming one):
//     p = u + be p ;  s = w + be s ;  x += al p ;  r -= al s       with u = r / diag, rounded by the caller
__device__ __forceinline__ void cg_cg_update(const float4& al, const float4& be, const float4& u, const float4& w, float4& x,
                                             float4& r, float4& p, float4& s) {
  p.x = fmaf(be.x, p.x, u.x); p.y = fmaf(be.y, p.y, u.y); p.z = fmaf(be.z, p.z, u.z); p.w = fmaf(be.w, p.w, u.w);
  s.x = fmaf(be.x, s.x, w.x); s.y = fmaf(be.y, s.y, w.y); s.z = fmaf(be.z, s.z, w.z); s.w = fmaf(be.w, s.w, w.w);
  x.x = fmaf(al.x, p.x, x.x); x.y = fmaf(al.y, p.y, x.y); x.z = fmaf(al.z, p.z, x.z); x.w = fmaf(al.w, p.w, x.w);
  r.x = fmaf(-al.x, s.x, r.x); r.y = fmaf(-al.y, s.y, r.y); r.z = fmaf(-al.z, s.z, r.z); r.w = fmaf(-al.w, s.w, r.w);
}

// alpha / beta of one live class column of the on-chip kernels, from g = <r,u> and d = <w,u> of this pass (T: the type of
// the reduced sums, fp32 in cg_small, fp64 in cg_resident and cg_cluster).  The quotients in fp32 (alpha and beta are fp32
// anyway), the cancellation-prone difference in fp64.  Approximate reciprocals (MUFU.RCP, deterministic): alpha and beta only
// have to be the SAME numbers in every CTA and in the x and r updates, their last bits do not matter to CG.  On breakdown
// (rounding at the fp32 floor) the column is frozen for good and al / be are left alone.
template <typename T, typename F>
__device__ __forceinline__ void cg_column_step(T g_new, T d_new, bool first, float& inv_g_old, float& inv_a_old, F& frozen, float& al,
                                               float& be) {
  const float bb = first ? 0.f : (float)g_new * inv_g_old;
  const double den = (double)d_new - (double)bb * (double)g_new * (double)inv_a_old;
  if (den > 0.0 && g_new > (T)0) {
    const float rg = __fdividef(1.f, (float)g_new);
    al = __fdividef((float)g_new, (float)den);
    be = bb;
    inv_a_old = (float)den * rg;
    inv_g_old = rg;
  } else {
    frozen = 1;
  }
}

// One thread, once per solve: iteration count, residual and status word.  Each kernel computes its residual its own way; the
// solve has converged when measure <= limit (compared only when the status is written).
template <typename T>
__device__ __forceinline__ void cg_write_stats(const CgSolve& P, int iters, float resid, bool bad, T measure, T limit) {
  if (P.iters_out) *P.iters_out = iters;
  if (P.resid_out) *P.resid_out = resid;
  if (P.status_out) {
    int st = 0;
    if (bad) st |= GLL_STATUS_NONFINITE;
    if (!bad && !(measure <= limit)) st |= GLL_STATUS_CG_NOT_CONVERGED;
    if (st) atomicOr(P.status_out, st);
  }
}

// right-hand side of class quad q of a row, from the padded fp32 array or straight from the caller's [m][l] array
__device__ __forceinline__ float4 cg_load_rhs4(const CgParams& P, int row, int q) {
  if (P.rhs_src == nullptr) return __ldg(reinterpret_cast<const float4*>(P.rhs + (size_t)row * P.lp + 4 * q));
  double sc = 1.0;
  if (P.rhs_scale != nullptr)
    sc = P.rhs_scale_f64 ? __ldg(reinterpret_cast<const double*>(P.rhs_scale)) : (double)__ldg(reinterpret_cast<const float*>(P.rhs_scale));
  float v[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int col = 4 * q + c;
    v[c] = 0.f;
    if (col < P.l)
      v[c] = (P.rhs_kind == 2) ? (float)(sc * __ldg(reinterpret_cast<const double*>(P.rhs_src) + (size_t)row * P.l + col))
                               : (float)(sc * (double)__ldg(reinterpret_cast<const float*>(P.rhs_src) + (size_t)row * P.l + col));
  }
  return make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void cg_store_copy4(const CgParams& P, int row, int q, const float4& x) {
  if (P.x_copy == nullptr) return;
  const float v[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int col = 4 * q + c;
    if (col < P.l) {
      if (P.x_copy_f64)
        reinterpret_cast<double*>(P.x_copy)[(size_t)row * P.l + col] = (double)v[c];
      else
        reinterpret_cast<float*>(P.x_copy)[(size_t)row * P.l + col] = v[c];
    }
  }
}

// The on-chip kernels.  *_fits(m, lp) is a host-only predicate (does the system fit the kernel's shared-memory and item
// budgets); *_launch runs a system that fits.  cg_pick decides which one runs.
// Multi-CTA kernel (cg_resident.cu): scratch must hold cg_resident_ws_bytes(m, lp) bytes.
size_t cg_resident_ws_bytes(int m, int lp);
bool cg_resident_fits(int m, int lp);
int cg_resident_launch(const CgParams& P, void* scratch, cudaStream_t st);
void cg_set_trace(void* buf);
void* cg_get_trace();
// One-CTA kernel for minibatch-sized systems (cg_small.cu).
bool cg_small_fits(int m, int lp);
int cg_small_launch(const CgParams& P, cudaStream_t st);
// Cluster kernel for the same minibatch-sized systems (cg_cluster.cu): one cluster of eight CTAs, exchanges through DSMEM.
bool cg_cluster_fits(int m, int lp);
int cg_cluster_launch(const CgParams& P, cudaStream_t st);

}  // namespace gll
