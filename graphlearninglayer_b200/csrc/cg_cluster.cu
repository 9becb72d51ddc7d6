// K4 for the minibatch-sized systems (C2/C3: 512 unlabeled rows x 10 classes; GLL.py:53 / GLL.py:93), organised for LATENCY.
// Same arithmetic as the other CG kernels (Jacobi-preconditioned Chronopoulos-Gear CG, per-column freeze and stop test of
// stable_conjgrad, GLL.py:247-276).  Such a solve is 6-10 iterations of a few thousand flops: what it costs is the length of
// the dependent chain per iteration.  A thread owns (row, class quad) ITEMS -- r, p, s in registers, x and w in shared memory --
// so that nothing in an iteration is longer than one row's edges (gathered four at a time) or one warp's share of a sum:
//   A  w = A u: an item walks its row's edges; u = r / diag lives in shared memory
//   B  <r,u>, <w,u>, <r,r>: per-item products to shared memory, one warp per (product, class quad, row part) adds its rows in
//      fp32 and finishes with one float4 butterfly; the partial sums (fp64) go into a slot per (CTA, part)
//   C  thread c adds the slots of class column c in a fixed order and derives alpha / beta; stop test
//   D  vector updates, new u
// ONE CLUSTER of eight CTAs of 320 threads runs systems of 64 to 2048 rows: a CTA owns an eighth of the rows, neighbour rows are
// gathered from the owner's shared memory (ld.shared::cluster, addresses precomputed with mapa), the partial sums are written
// into a slot of EVERY CTA's shared memory (st.shared::cluster) and two barrier.cluster per iteration replace the two grid
// barriers of the multi-CTA kernel (cg_resident.cu: 1.2 us each through L2).  No global-memory traffic inside the loop.
// It takes a system when cg_pick routes it here (a sparsity hint of at most 5 entries per row, or GLL_B200_CG_PATH=cluster)
// and its items (class quads x rows per CTA) fit four per thread; the others go to cg_small.cu or cg_resident.cu.
#include <math.h>
#include <string.h>

#include "cg_common.cuh"

namespace gll {
namespace {

constexpr int CC_CTAS = 8;
// (256 / 320 / 384 threads per CTA measured the same at C2, 2.95-3.2 us per iteration; the same item layout on ONE CTA: 3.8 us
//  with 512 threads, 5.0 us with 1024 (spills at 64 registers) -- an iteration is ~450 mostly dependent instructions per warp,
//  and what the cluster buys is a shorter chain per warp, not bandwidth)
constexpr int CC_THREADS = 320;
constexpr int CC_WARPS = CC_THREADS / 32;
constexpr int CC_MAX_NIT = 4;
constexpr size_t CC_SMEM_BUDGET = 208 * 1024;  // (512 rows x 12 class columns on one CTA: 145 KB of vectors and products)

__device__ __forceinline__ uint32_t cc_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cc_sync() {  // everybody in the cluster is here, and their shared-memory writes are visible
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// cluster-window address of the same shared-memory offset in CTA `rank` (a CTA's own shared::cta addresses are valid there too)
__device__ __forceinline__ uint32_t cc_mapa(uint32_t local, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
  return r;
}
__device__ __forceinline__ float4 cc_ld4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void cc_st_f64(uint32_t addr, double v) {
  asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}

struct CcShape {
  int R;         // rows per CTA (a multiple of 32)
  int nparts;    // row parts per (product, class quad) sum
  int part_rows; // rows per part (a multiple of 32)
  int edge_cap;  // edges of a CTA's slice that fit in shared memory
};

template <int NIT>
__global__ void __launch_bounds__(CC_THREADS, 1) cg_cluster_kernel(CgParams P, CcShape S, unsigned long long* trace) {
  // debug timeline (gll_debug_cg_trace, tools/cg_small_trace.py): trace[pass * 8 + phase] = SM clock of CTA 0, thread 0
#define CC_STAMP(phase) do { if (trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0 && iter < 15) trace[iter * 8 + (phase)] = (unsigned long long)clock64(); } while (0)
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const int lp = P.lp, Q = lp >> 2, m = P.m, E3 = 3 * lp, R = S.R;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) trace[15 * 8 + 7] = (unsigned long long)clock64();  // kernel entry
  const int rank = (int)cc_rank();
  const int row0 = rank * R, rows = max(0, min(R, m - row0));  // my rows (R = rows per CTA, the same in every CTA)
  const int nslots = CC_CTAS * S.nparts;
  // ---- shared memory (identical layout in every CTA: remote addresses are local offsets mapped with mapa) ----
  float* us = reinterpret_cast<float*>(sm_raw);                              // [R][lp]   u = r / diag of my rows
  float4* prod = reinterpret_cast<float4*>(us + (size_t)R * lp);             // [3][Q][R] r*u, w*u, r*r per item
  float4* xs = prod + (size_t)3 * Q * R;                                     // [Q][R] x per item
  float4* ws = xs + (size_t)Q * R;                                           // [Q][R] w per item
  double* part = reinterpret_cast<double*>(ws + (size_t)Q * R);              // [nslots][E3] slot (c, part): partial sums
  double* red = part + (size_t)nslots * E3;                                  // [E3] sums over all rows
  float* alpha = reinterpret_cast<float*>(red + E3);                         // [lp]
  float* beta = alpha + lp;                                                  // [lp]
  int* flags = reinterpret_cast<int*>(beta + lp);                            // [4] live / bad of this pass
  int* lptr = flags + 4;                                                     // [R + 1]
  uint32_t* eaddr = reinterpret_cast<uint32_t*>(lptr + (R + 1));             // [edge_cap] (cluster) address of the edge's u row
  float* eval = reinterpret_cast<float*>(eaddr + S.edge_cap);                // [edge_cap]

  const uint32_t us_s = cc_smem_u32(us), part_s = cc_smem_u32(part);
  auto u_row_addr = [&](int j) {
    const int owner = j / R;
    return cc_mapa(us_s + (uint32_t)((j - owner * R) * lp) * 4u, (uint32_t)owner);
  };
  const int e_begin = (rows > 0) ? __ldg(P.ptr + row0) : 0;
  const int nnz = (rows > 0) ? __ldg(P.ptr + row0 + rows) - e_begin : 0;
  const bool cached = nnz <= S.edge_cap;  // (always at minibatch sizes; otherwise the edges are read from global memory)
  for (int i = tid; i <= rows; i += CC_THREADS) lptr[i] = __ldg(P.ptr + row0 + i) - e_begin;
  if (cached)
    for (int e = tid; e < nnz; e += CC_THREADS) {
      eaddr[e] = u_row_addr(__ldg(P.col + e_begin + e));
      eval[e] = __ldg(P.val + e_begin + e);
    }

  // ---- my items (quad-major inside the CTA: item = quad * R + local row): x = 0, r = b, p = s = 0 ----
  int lrow[NIT], quad[NIT];
  bool on[NIT];
  float dg[NIT], dinv[NIT];
  float4 r[NIT], p[NIT], s[NIT];
#pragma unroll
  for (int k = 0; k < NIT; ++k) {
    const int it = tid + k * CC_THREADS;
    quad[k] = it / R;
    lrow[k] = it - quad[k] * R;
    on[k] = quad[k] < Q && lrow[k] < rows;
    dg[k] = on[k] ? __ldg(P.diag + row0 + lrow[k]) : 1.f;
    dinv[k] = on[k] ? 1.f / dg[k] : 0.f;
    r[k] = on[k] ? cg_load_rhs4(P, row0 + lrow[k], quad[k]) : zero4();
    p[k] = s[k] = zero4();
    if (quad[k] < Q) {
      xs[(size_t)quad[k] * R + lrow[k]] = zero4();
      *reinterpret_cast<float4*>(us + (size_t)lrow[k] * lp + 4 * quad[k]) = scale4(r[k], dinv[k]);
    }
  }
  // per-column CG scalars: thread c owns class column c (every CTA computes identical values)
  float inv_g_old = 1.f, inv_a_old = 1.f;
  bool frozen = false;
  double tol2 = 0.0;
  int iter = 0;
  bool bad_any = false;
  cc_sync();  // every CTA's u and edge addresses are in place

  while (true) {
    CC_STAMP(0);
    // ================= A: w = A u and the per-item products =================
#pragma unroll
    for (int k = 0; k < NIT; ++k) {
      if (quad[k] < Q) {
        float4 a = zero4();
        if (on[k]) {
          const int e1 = lptr[lrow[k] + 1];
          const uint32_t qoff = 16u * (uint32_t)quad[k];
          int e = lptr[lrow[k]];
          if (cached) {
            // four neighbour rows in flight (a remote row is ~215 cycles away, a local one ~30; one at a time made this phase
            // the longest of the iteration)
            for (; e + 4 <= e1; e += 4) {
              const uint32_t a0 = eaddr[e], a1 = eaddr[e + 1], a2 = eaddr[e + 2], a3 = eaddr[e + 3];
              const float4 u0 = cc_ld4(a0 + qoff), u1 = cc_ld4(a1 + qoff), u2 = cc_ld4(a2 + qoff), u3 = cc_ld4(a3 + qoff);
              fma4(a, eval[e], u0);
              fma4(a, eval[e + 1], u1);
              fma4(a, eval[e + 2], u2);
              fma4(a, eval[e + 3], u3);
            }
            if (e + 2 <= e1) {
              const uint32_t a0 = eaddr[e], a1 = eaddr[e + 1];
              const float4 u0 = cc_ld4(a0 + qoff), u1 = cc_ld4(a1 + qoff);
              fma4(a, eval[e], u0);
              fma4(a, eval[e + 1], u1);
              e += 2;
            }
            if (e < e1) fma4(a, eval[e], cc_ld4(eaddr[e] + qoff));
          } else {
            for (; e < e1; ++e) fma4(a, __ldg(P.val + e_begin + e), cc_ld4(u_row_addr(__ldg(P.col + e_begin + e)) + qoff));
          }
        }
        const float4 u4 = scale4(r[k], dinv[k]);
        const float4 w4 = on[k] ? make_float4(fmaf(dg[k], u4.x, -a.x), fmaf(dg[k], u4.y, -a.y), fmaf(dg[k], u4.z, -a.z), fmaf(dg[k], u4.w, -a.w))
                                : zero4();
        const size_t o = (size_t)quad[k] * R + lrow[k];
        ws[o] = w4;
        prod[o] = make_float4(r[k].x * u4.x, r[k].y * u4.y, r[k].z * u4.z, r[k].w * u4.w);
        prod[(size_t)Q * R + o] = make_float4(w4.x * u4.x, w4.y * u4.y, w4.z * u4.z, w4.w * u4.w);
        prod[(size_t)2 * Q * R + o] = make_float4(r[k].x * r[k].x, r[k].y * r[k].y, r[k].z * r[k].z, r[k].w * r[k].w);
      }
    }
    CC_STAMP(4);
    if (tid == 0) flags[0] = 0;
    __syncthreads();
    // ================= B: partial sums, one warp per (product, class quad, row part), into a slot of EVERY CTA =================
#pragma unroll 1
    for (int sj = warp; sj < 3 * Q * S.nparts; sj += CC_WARPS) {
      const int job = sj / S.nparts, pt = sj - job * S.nparts;
      const float4* src = prod + (size_t)job * R;
      const int i1 = min(R, (pt + 1) * S.part_rows);
      float4 f = zero4();  // fp32 inside a part (<= a few hundred rows, as in the former one-CTA kernel), fp64 across parts and CTAs
      for (int i = pt * S.part_rows + lane; i < i1; i += 32) {  // rows beyond `rows` hold zeros (items that are not `on`)
        const float4 v = src[i];
        f.x += v.x; f.y += v.y; f.z += v.z; f.w += v.w;
      }
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) {  // four independent chains
        f.x += __shfl_xor_sync(FULL, f.x, o);
        f.y += __shfl_xor_sync(FULL, f.y, o);
        f.z += __shfl_xor_sync(FULL, f.z, o);
        f.w += __shfl_xor_sync(FULL, f.w, o);
      }
      // lane c < CC_CTAS sends the four sums to CTA c (job = v * Q + quad  ->  element v * lp + 4 * quad + j)
      if (lane < CC_CTAS) {
        const int v = job / Q, qd = job - v * Q;
        const uint32_t off = part_s + (uint32_t)((rank * S.nparts + pt) * E3 + v * lp + 4 * qd) * 8u;
        const uint32_t dst = cc_mapa(off, (uint32_t)lane);
        cc_st_f64(dst, (double)f.x);
        cc_st_f64(dst + 8u, (double)f.y);
        cc_st_f64(dst + 16u, (double)f.z);
        cc_st_f64(dst + 24u, (double)f.w);
      }
    }
    CC_STAMP(5);
    cc_sync();  // (1) all partial sums have landed
    CC_STAMP(1);
    if (tid < E3) {
      double t = 0.0;
      for (int c = 0; c < nslots; ++c) t += part[(size_t)c * E3 + tid];  // the same order in every CTA
      red[tid] = t;
    }
    __syncthreads();
    CC_STAMP(2);
    // ================= C: scalars =================
    if (iter == 0) {
      double mx = 0.0;
      for (int c = 0; c < lp; ++c) mx = fmax(mx, red[2 * lp + c]);
      tol2 = (P.tol < 0.f) ? (double)P.tol * (double)P.tol * mx : (double)P.tol * (double)P.tol;
    }
    int live = 0, bad = 0;
    if (tid < lp) {
      const double g_new = red[tid], d_new = red[lp + tid], rr = red[2 * lp + tid];
      bad = (!(rr == rr) || rr > 1.0e300) ? 1 : 0;
      float al = 0.f, be = 0.f;
      if (!frozen && rr > tol2) {
        live = 1;
        cg_column_step(g_new, d_new, iter == 0, inv_g_old, inv_a_old, frozen, al, be);
      }
      alpha[tid] = al;
      beta[tid] = be;
    }
    if (live | bad) atomicOr(&flags[0], live | (bad << 1));
    __syncthreads();
    const int fl = flags[0];
    CC_STAMP(3);
    bad_any = (fl & 2) != 0;
    if (bad_any || !(fl & 1) || iter >= P.max_iter) break;  // identical decision in every CTA: the sums are identical
    ++iter;
    // ================= D: vector updates, publish the new u =================
#pragma unroll
    for (int k = 0; k < NIT; ++k) {
      if (quad[k] < Q) {
        const float4 al = *reinterpret_cast<const float4*>(alpha + 4 * quad[k]);
        const float4 be = *reinterpret_cast<const float4*>(beta + 4 * quad[k]);
        const float di = dinv[k];
        const size_t o = (size_t)quad[k] * R + lrow[k];
        float4 x4 = xs[o];
        cg_cg_update(al, be, scale4(r[k], di), ws[o], x4, r[k], p[k], s[k]);
        xs[o] = x4;
        *reinterpret_cast<float4*>(us + (size_t)lrow[k] * lp + 4 * quad[k]) = scale4(r[k], di);
      }
    }
    CC_STAMP(6);
    cc_sync();  // (2) the new u is visible to everybody; the slots of `part` may be rewritten
  }
#undef CC_STAMP

#pragma unroll
  for (int k = 0; k < NIT; ++k)
    if (on[k]) {
      const float4 x4 = xs[(size_t)quad[k] * R + lrow[k]];
      *reinterpret_cast<float4*>(P.x + (size_t)(row0 + lrow[k]) * lp + 4 * quad[k]) = x4;
      cg_store_copy4(P, row0 + lrow[k], quad[k], x4);
    }
  if (rank == 0 && tid == 0) {
    double mx = 0.0;
    for (int c = 0; c < lp; ++c) mx = fmax(mx, red[2 * lp + c]);
    cg_write_stats(P, iter, (float)sqrt(mx), bad_any, mx, tol2);
  }
  cc_sync();  // nobody exits while a peer may still read its u rows or write into its slots
}

size_t cc_fixed_smem(int R, int lp, int nslots) {
  const int Q = lp >> 2, E3 = 3 * lp;
  size_t b = sizeof(float) * (size_t)R * lp + 16 * (size_t)5 * Q * R + sizeof(double) * ((size_t)nslots * E3 + E3) +
             sizeof(float) * 2 * (size_t)lp + sizeof(int) * (4 + (size_t)R + 1);
  return align_up(b, 16);
}

struct CcPlan {
  int nit;  // items per thread; 0: the system does not fit
  CcShape S;
  size_t smem;
};

CcPlan cluster_plan(int m, int lp) {
  CcPlan p = {};
  if (m < 64 || m > 2048) return p;  // below 64 rows there is nothing to share
  const int Q = lp >> 2;
  CcShape& S = p.S;
  S.R = ceil_div(ceil_div(m, CC_CTAS), 32) * 32;  // whole warps of rows per class quad
  const int nit = (int)(((long long)Q * S.R + CC_THREADS - 1) / CC_THREADS);
  if (nit > CC_MAX_NIT) return p;
  S.nparts = max(1, min(CC_WARPS / (3 * Q), S.R / 32));  // use the warps that the (product, quad) jobs leave idle
  S.part_rows = ceil_div(ceil_div(S.R, S.nparts), 32) * 32;
  const size_t fixed = cc_fixed_smem(S.R, lp, CC_CTAS * S.nparts);
  if (fixed + 16384 > CC_SMEM_BUDGET) return p;
  S.edge_cap = (int)((CC_SMEM_BUDGET - fixed) / 8);
  p.smem = fixed + (size_t)S.edge_cap * 8;
  p.nit = nit;
  return p;
}

}  // namespace

bool cg_cluster_fits(int m, int lp) { return cluster_plan(m, lp).nit > 0; }

int cg_cluster_launch(const CgParams& P, cudaStream_t st) {
  static const void* const kernels[CC_MAX_NIT] = {(const void*)cg_cluster_kernel<1>, (const void*)cg_cluster_kernel<2>,
                                                  (const void*)cg_cluster_kernel<3>, (const void*)cg_cluster_kernel<4>};
  CcPlan pl = cluster_plan(P.m, P.lp);
  const void* kern = kernels[pl.nit - 1];
  GLL_CUDA_CHECK(set_max_dynamic_smem_once(kern, (int)CC_SMEM_BUDGET));
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(CC_CTAS);
  cfg.blockDim = dim3(CC_THREADS);
  cfg.dynamicSmemBytes = pl.smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CC_CTAS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CgParams Pc = P;
  unsigned long long* trace = (unsigned long long*)cg_get_trace();
  void* args[] = {&Pc, &pl.S, &trace};
  GLL_PROF(KID_CG, st);
  GLL_CUDA_CHECK(cudaLaunchKernelExC(&cfg, kern, args));
  return GLL_OK;
}

}  // namespace gll
