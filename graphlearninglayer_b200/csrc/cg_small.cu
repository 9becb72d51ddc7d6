// K4, one-CTA variant for the minibatch-sized systems (C2/C3: 512 unlabeled rows x 10 classes; GLL.py:53 / GLL.py:93).
// Same arithmetic as cg_resident.cu (Jacobi-preconditioned Chronopoulos-Gear CG, per-column freeze and stop test of
// stable_conjgrad, GLL.py:247-276), organised for LATENCY: such a solve is 6-10 iterations of a few thousand flops,
// so what it costs is the length of the dependent chain per iteration, not bandwidth.
//   * every thread owns up to NIT (row, class quad) items and keeps x, r, p, s, w of them in REGISTERS for the whole solve;
//     only u = r/diag lives in shared memory (the SpMV gathers it)
//   * items are quad-major and the (power-of-two) padded row count divides the CTA size: all items of a thread belong to one
//     row, whose edges are walked once for all class quads
//   * dot products: per-item products go to shared memory, one warp per (dot, quad) adds the rows (independent loads) and
//     finishes with ONE butterfly -- warp shuffles run at ~0.5 per clock per SM, a butterfly per item was 3 us per iteration
//   * warp 0 derives alpha / beta / stop; four __syncthreads per iteration
#include <math.h>

#include "cg_common.cuh"

namespace gll {
namespace {

constexpr int CS_THREADS = 512;
constexpr int CS_WARPS = CS_THREADS / 32;
constexpr int CS_MAX_NIT = 4;
constexpr size_t CS_SMEM_BUDGET = 160 * 1024;

__device__ __forceinline__ float4 f4mul(const float4& a, const float4& b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float4 f4butterfly(float4 a) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    a.x += __shfl_xor_sync(FULL, a.x, o);
    a.y += __shfl_xor_sync(FULL, a.y, o);
    a.z += __shfl_xor_sync(FULL, a.z, o);
    a.w += __shfl_xor_sync(FULL, a.w, o);
  }
  return a;
}
// explicit shared-space 128-bit load from a 32-bit shared address (the generic form makes the compiler re-derive the
// shared window with an S2R inside the gather loop)
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

template <int NIT>
__global__ void __launch_bounds__(CS_THREADS, 1) cg_small_kernel(CgParams P, int rows_pad, int csr_cap, unsigned long long* trace) {
  // debug timeline (gll_debug_cg_trace): trace[pass * 8 + phase] = SM cycle counter, thread 0
#define CS_STAMP(phase) do { if (trace != nullptr && threadIdx.x == 0 && iter < 16) trace[iter * 8 + (phase)] = (unsigned long long)clock64(); } while (0)
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const int lp = P.lp, Q = lp >> 2, m = P.m;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* us = reinterpret_cast<float*>(sm_raw);                              // [rows_pad][lp]   u = r / diag
  float4* prod = reinterpret_cast<float4*>(us + (size_t)rows_pad * lp);       // [3][Q][rows_pad] r*u, w*u, r*r per item
  float* red = reinterpret_cast<float*>(prod + (size_t)3 * Q * rows_pad);     // [3][lp]  <r,u>, <w,u>, <r,r>
  float* alpha = red + 3 * lp;                                                // [lp]
  float* beta = alpha + lp;                                                   // [lp]
  int* stop_s = reinterpret_cast<int*>(beta + lp);                            // [4]
  int* lptr = stop_s + 4;                                                     // [m + 1]
  int* ccol = lptr + (m + 1);                                                 // [csr_cap]
  float* cval = reinterpret_cast<float*>(ccol + csr_cap);                     // [csr_cap]

  if (trace != nullptr && threadIdx.x == 0) trace[15 * 8 + 7] = (unsigned long long)clock64();  // kernel entry
  const int nnz = __ldg(P.ptr + m);
  const bool cached = nnz <= csr_cap;
  for (int i = tid; i <= m; i += CS_THREADS) lptr[i] = __ldg(P.ptr + i);
  if (cached)
    for (int e = tid; e < nnz; e += CS_THREADS) {
      ccol[e] = __ldg(P.col + e);
      cval[e] = __ldg(P.val + e);
    }

  // ---- my items (quad-major: item = quad * rows_pad + row): x = 0, r = b, p = s = 0 ----
  int row[NIT], quad[NIT], uoff[NIT];
  bool on[NIT];
  float dg[NIT], dinv[NIT];
  float4 x[NIT], r[NIT], p[NIT], s[NIT], w[NIT];
#pragma unroll
  for (int k = 0; k < NIT; ++k) {
    const int it = tid + k * CS_THREADS;
    quad[k] = it / rows_pad;
    row[k] = it - quad[k] * rows_pad;
    on[k] = quad[k] < Q && row[k] < m;
    dg[k] = on[k] ? __ldg(P.diag + row[k]) : 1.f;
    dinv[k] = on[k] ? 1.f / dg[k] : 0.f;
    r[k] = on[k] ? cg_load_rhs4(P, row[k], quad[k]) : zero4();
    x[k] = p[k] = s[k] = w[k] = zero4();
    uoff[k] = (quad[k] < Q) ? 4 * quad[k] : 0;
    if (quad[k] < Q) *reinterpret_cast<float4*>(us + (size_t)row[k] * lp + 4 * quad[k]) = scale4(r[k], dinv[k]);
  }
  // per-column CG scalars live in warp 0: lane owns columns lane, lane + 32, ...
  constexpr int CPL = CG_MAX_LP / 32;
  float inv_g_old[CPL], inv_a_old[CPL];
  bool frozen[CPL];
#pragma unroll
  for (int j = 0; j < CPL; ++j) {
    inv_g_old[j] = inv_a_old[j] = 1.f;
    frozen[j] = false;
  }
  uint32_t us_s;
  {
    unsigned long long t;
    asm volatile("cvta.to.shared.u64 %0, %1;" : "=l"(t) : "l"(us));
    us_s = (uint32_t)t;
  }
  float tol2 = 0.f, mx_all = 0.f;
  int iter = 0;
  bool bad = false;
  __syncthreads();

  while (true) {
    CS_STAMP(0);
    // ================= A: w = A u and the per-item products =================
    // rows_pad divides the CTA size, so all items of a thread belong to ONE row: its edges are walked once for all quads
    {
      float4 a[NIT];
#pragma unroll
      for (int k = 0; k < NIT; ++k) a[k] = zero4();
      // no branches inside the edge loop (items beyond the last quad gather quad 0 and are discarded below), and one
      // copy per address space of the CSR: otherwise every gather re-derives the shared-memory window (S2UR in the loop)
      auto walk = [&](const int* __restrict__ cj, const float* __restrict__ cv) {
        const int e1 = lptr[row[0] + 1];
        int e = lptr[row[0]];
        if (trace != nullptr && threadIdx.x == 0 && iter < 15) trace[iter * 8 + 7] = (unsigned long long)clock64() + (unsigned long long)((e + e1) & 0);
#pragma unroll 2
        for (; e < e1; ++e) {
          const float we = cv[e];
          const uint32_t uj = us_s + (uint32_t)(cj[e] * lp) * 4u;
#pragma unroll
          for (int k = 0; k < NIT; ++k) fma4(a[k], we, lds128(uj + 4u * (uint32_t)uoff[k]));
        }
      };
      if (row[0] < m) {
        if (cached)
          walk(ccol, cval);
        else
          walk(P.col, P.val);
      }
      CS_STAMP(4);
#pragma unroll
      for (int k = 0; k < NIT; ++k) {
        if (quad[k] < Q) {
          const float4 u4 = scale4(r[k], dinv[k]);
          w[k] = make_float4(fmaf(dg[k], u4.x, -a[k].x), fmaf(dg[k], u4.y, -a[k].y), fmaf(dg[k], u4.z, -a[k].z),
                             fmaf(dg[k], u4.w, -a[k].w));
          if (!on[k]) w[k] = zero4();
          const size_t o = (size_t)quad[k] * rows_pad + row[k];
          prod[o] = f4mul(r[k], u4);
          prod[(size_t)Q * rows_pad + o] = f4mul(w[k], u4);
          prod[(size_t)2 * Q * rows_pad + o] = f4mul(r[k], r[k]);
        }
      }
    }
    CS_STAMP(5);
    if (trace != nullptr && threadIdx.x == CS_THREADS - 1 && iter < 16) trace[iter * 8 + 6] = (unsigned long long)clock64();
    __syncthreads();
    CS_STAMP(1);
    // ================= B: one warp per (dot, quad): rows summed serially per lane, then ONE butterfly =================
#pragma unroll 1
    for (int job = warp; job < 3 * Q; job += CS_WARPS) {
      const float4* src = prod + (size_t)job * rows_pad;
      float4 t0 = zero4(), t1 = zero4();
#pragma unroll 4
      for (int i = lane; i < rows_pad; i += 64) {
        const float4 v0 = src[i];
        const float4 v1 = (i + 32 < rows_pad) ? src[i + 32] : zero4();
        t0.x += v0.x; t0.y += v0.y; t0.z += v0.z; t0.w += v0.w;
        t1.x += v1.x; t1.y += v1.y; t1.z += v1.z; t1.w += v1.w;
      }
      t0.x += t1.x; t0.y += t1.y; t0.z += t1.z; t0.w += t1.w;
      t0 = f4butterfly(t0);
      if (lane == 0) *reinterpret_cast<float4*>(red + (job / Q) * lp + 4 * (job % Q)) = t0;
    }
    __syncthreads();
    CS_STAMP(2);
    // ================= C: scalars (warp 0) =================
    if (warp == 0) {
      float rrc[CPL];
      float mx = 0.f, mx_live = 0.f;
      int badi = 0;
#pragma unroll
      for (int j = 0; j < CPL; ++j) {
        const int c = lane + 32 * j;
        rrc[j] = (c < lp) ? red[2 * lp + c] : 0.f;
        badi |= (!(rrc[j] == rrc[j]) || rrc[j] > 3.0e38f) ? 1 : 0;
        mx = fmaxf(mx, rrc[j]);
        if (!frozen[j]) mx_live = fmaxf(mx_live, rrc[j]);
      }
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, o));
        mx_live = fmaxf(mx_live, __shfl_xor_sync(FULL, mx_live, o));
        badi |= __shfl_xor_sync(FULL, badi, o);
      }
      if (iter == 0) tol2 = (P.tol < 0.f) ? P.tol * P.tol * mx : P.tol * P.tol;
      bad = badi != 0;
      mx_all = mx;
      const bool stop = bad || mx_live <= tol2 || iter >= P.max_iter;
      if (lane == 0) stop_s[0] = stop ? 1 : 0;
      if (!stop) {
#pragma unroll
        for (int j = 0; j < CPL; ++j) {
          const int c = lane + 32 * j;
          if (c < lp) {
            const float g_new = red[c], d_new = red[lp + c];
            float al = 0.f, be = 0.f;
            // (approximate reciprocals: three IEEE divisions in this one-warp section cost ~0.2 us per pass)
            if (!frozen[j] && rrc[j] > tol2) cg_column_step(g_new, d_new, iter == 0, inv_g_old[j], inv_a_old[j], frozen[j], al, be);
            alpha[c] = al;
            beta[c] = be;
          }
        }
      }
    }
    __syncthreads();
    CS_STAMP(3);
    if (stop_s[0]) break;
    ++iter;
    // ================= D: vector updates in registers, publish the new u =================
#pragma unroll
    for (int k = 0; k < NIT; ++k) {
      if (quad[k] < Q) {
        const float4 al = *reinterpret_cast<const float4*>(alpha + 4 * quad[k]);
        const float4 be = *reinterpret_cast<const float4*>(beta + 4 * quad[k]);
        const float di = dinv[k];
        cg_cg_update(al, be, scale4(r[k], di), w[k], x[k], r[k], p[k], s[k]);
        *reinterpret_cast<float4*>(us + (size_t)row[k] * lp + 4 * quad[k]) = scale4(r[k], di);
      }
    }
    __syncthreads();
  }
#undef CS_STAMP

#pragma unroll
  for (int k = 0; k < NIT; ++k)
    if (on[k]) {
      *reinterpret_cast<float4*>(P.x + (size_t)row[k] * lp + 4 * quad[k]) = x[k];
      cg_store_copy4(P, row[k], quad[k], x[k]);
    }
  if (tid == 0) cg_write_stats(P, iter, sqrtf(mx_all), bad, mx_all, tol2);  // warp 0 holds the stop state
}

struct CsPlan {
  int nit;  // items per thread; 0: the system does not fit
  int rows_pad, csr_cap;
  size_t smem;
};

CsPlan small_plan(int m, int lp) {
  CsPlan p = {};
  if (m > CS_THREADS) return p;
  p.rows_pad = 32;  // a power of two, so that it divides the CTA size: every thread's items then share their row
  while (p.rows_pad < m) p.rows_pad <<= 1;
  const int Q = lp >> 2;
  const int nit = (int)(((long long)Q * p.rows_pad + CS_THREADS - 1) / CS_THREADS);
  if (nit > CS_MAX_NIT) return p;
  const size_t fixed = sizeof(float) * (size_t)p.rows_pad * lp + 16 * (size_t)3 * Q * p.rows_pad + sizeof(float) * 5 * (size_t)lp + 16 +
                       sizeof(int) * ((size_t)m + 1) + 64;
  if (fixed + 4096 > CS_SMEM_BUDGET) return p;
  p.csr_cap = (int)((CS_SMEM_BUDGET - fixed) / 8);
  p.smem = fixed + (size_t)p.csr_cap * 8;
  p.nit = nit;
  return p;
}

}  // namespace

bool cg_small_fits(int m, int lp) { return small_plan(m, lp).nit > 0; }

int cg_small_launch(const CgParams& P, cudaStream_t st) {
  static const void* const kernels[CS_MAX_NIT] = {(const void*)cg_small_kernel<1>, (const void*)cg_small_kernel<2>,
                                                  (const void*)cg_small_kernel<3>, (const void*)cg_small_kernel<4>};
  CsPlan pl = small_plan(P.m, P.lp);
  const void* kern = kernels[pl.nit - 1];
  GLL_CUDA_CHECK(set_max_dynamic_smem_once(kern, (int)CS_SMEM_BUDGET));
  CgParams Pc = P;
  unsigned long long* trace = (unsigned long long*)cg_get_trace();
  void* args[] = {&Pc, &pl.rows_pad, &pl.csr_cap, &trace};
  GLL_PROF(KID_CG, st);
  GLL_CUDA_CHECK(cudaLaunchKernel(kern, dim3(1), dim3(CS_THREADS), args, pl.smem, st));
  return GLL_OK;
}

}  // namespace gll
