// K4, on-chip variant -- multi-right-hand-side Jacobi-preconditioned CG whose state never leaves the SM.
// (replaces spsolve at GLL.py:53 / GLL.py:93; stopping rule and per-column freeze of stable_conjgrad, GLL.py:247-276)
//
// Every CTA owns a block of rows for the whole solve and keeps x, r, p, s = Ap, w = Au (u = r/diag), 1/diag and its slice
// of the matrix in SHARED MEMORY across iterations.  The only global traffic per iteration is
//   * the preconditioned residual u, published by its owner and gathered by the CTAs whose rows reference it (L2), and
//   * 3*l dot-product partials per CTA (fp64).
// Recurrences are Chronopoulos-Gear's single-reduction CG (one SpMV, one reduction of <r,u>, <w,u>, <r,r> per iteration):
//     p = u + b p ;  s = w + b s ;  x += a p ;  r -= a s ;  u = r/diag ;  w = A u
//     b = g'/g ,  a = g' / (d - b g'/a_old)      with g = <r,u>, d = <w,u>
// (the pipelined variant that hides the reduction behind the SpMV was tried in an fp32 model of this system and does not
// reach the 1e-7 residual: its recurrences for u and w drift, profiles/r02_cg_trace.md).
//
// What an iteration costs on 148 SMs is latency, not bandwidth (a C4-size system, 14336 rows x 10 classes, is 97 rows
// per CTA), so the kernel is organised around the measured costs (tools/xchg_bench.cu, profiles/r02a_xchg_bench.txt):
//   * one L2 hop between two SMs is ~450 ns; a grid barrier through ONE atomic counter (red.release + ld.acquire spin by
//     one thread per CTA) costs 1.2 us with 148 CTAs -- cheaper than any mailbox scheme (4-5 us), so both exchanges of an
//     iteration are a counter barrier: (B) "u is published", (A) "dot-product partials are written".  After (A) every CTA
//     reads all G x 3l partials with coalesced loads and adds them in the same fixed order, so all CTAs take identical
//     branches and the result is bit-reproducible (no floating-point atomics).
//   * the SpMV is bound by the L1TEX wavefront rate (one 128-byte line per gathered row of u: ~2 us for the 2.5 k gathers
//     of a CTA), so it issues exactly one gather per edge and nothing else: rows are cut into SEGMENTS of 10 edges
//     (built once per solve in shared memory), a thread owns one (segment, class quad) and has its 10 loads in flight at
//     once -- no idle lanes for short rows, no tail for hub rows (degree 91 against a mean of 26) -- and u rows of 48
//     bytes are stored with a 64-byte stride so that no gather straddles a line.  Segment sums are added per row in a
//     second, shared-memory-only pass.
//   * the three dot products take one warp per (product, class column) with ONE butterfly each.
// With a single CTA (systems of a few hundred rows) the exchanges degenerate to __syncthreads and u stays in shared memory.
#include <math.h>

#include "cg_common.cuh"

namespace gll {
namespace {

constexpr int CR_THREADS = 1024;
constexpr int CR_WARPS = CR_THREADS / 32;
// Edges per segment = independent gathers in flight per thread.  10 makes the C4-size system (97 rows x ~26 edges x 3
// class quads per CTA) exactly one round of <= 1024 (segment, quad) tasks; with 8 it is 1092 tasks = a second, nearly
// empty round that costs a full L2 round trip.
constexpr int CR_SEG = 10;
constexpr size_t CR_SMEM_BUDGET = 200 * 1024;
constexpr int CR_MAX_GRID = 160;  // the sum over CTAs keeps CR_MAX_GRID / 32 loads per lane in flight

struct CrParams {
  CgParams cg;
  float* ubuf;        // [m][ustride] published u
  double* part;       // [3*lp][grid] dot-product partials of every CTA (column-major)
  unsigned* counter;  // grid barrier (zeroed before the launch)
  int rows_cap;       // rows per CTA
  int seg_cap;        // segments a CTA can hold in shared memory
  int ustride;        // floats per row of ubuf
  unsigned long long* trace;  // debug: [grid][16 passes][16 phases] clock64 stamps (NULL = off)
};

__device__ __forceinline__ void red_release_add_u32(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// All CTAs are co-resident (cooperative launch).  The release of thread 0 is cumulative over the CTA's earlier stores
// (ordered before it by bar.sync), the acquire + bar.sync order every thread's later loads after the peers' stores.
__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    red_release_add_u32(counter, 1u);
    while (ld_acquire_u32(counter) < target) {
    }
  }
  __syncthreads();
}

// debug timeline (TRACE instantiation only).  BAR.SYNC is deferred-blocking (a clock read right behind it can run before the barrier releases), so
// the stamp first touches shared memory, which waits for the barrier.
__device__ __forceinline__ void cr_stamp(const CrParams& R, int pass, int phase) {
  if (R.trace != nullptr && threadIdx.x == 0 && pass < 16) {
    unsigned dummy;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(dummy) : "r"(0u) : "memory");
    unsigned long long t;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(t) : "r"(dummy) : "memory");
    R.trace[((size_t)blockIdx.x * 16 + pass) * 16 + phase] = t;
  }
}

struct Ctrl {
  double tol2;  // squared absolute tolerance, fixed in pass 0
  int flags;    // bit 0: some column still moves, bit 1: non-finite residual (set by the column threads, cleared every pass)
  int pad;
};

// Rare path: a row block whose segments do not fit in shared memory walks the CSR in global memory, one thread per
// (row, class quad).
template <bool SINGLE>
__device__ __forceinline__ void spmv_rows_from_global(const CgParams& P, int row0, int rows, const float* ub, int ust, const float* rs,
                                                   float* ws, const float* dg, const float* dinv) {
  const int lp = P.lp, Q = lp >> 2;
#pragma unroll 1
  for (int it = threadIdx.x; it < rows * Q; it += CR_THREADS) {
    const int i = it / Q, q = it - i * Q;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    const int e1 = __ldg(P.ptr + row0 + i + 1);
#pragma unroll 1
    for (int e = __ldg(P.ptr + row0 + i); e < e1; ++e) {
      const int j = __ldg(P.col + e);
      const float4 uj = SINGLE ? *reinterpret_cast<const float4*>(ub + (size_t)j * ust + 4 * q) : ldcg4(ub + (size_t)j * ust + 4 * q);
      fma4(a, __ldg(P.val + e), uj);
    }
    const size_t o = (size_t)i * lp + 4 * q;
    const float4 u4 = scale4(*reinterpret_cast<const float4*>(rs + o), dinv[i]);
    const float dgi = dg[i];
    *reinterpret_cast<float4*>(ws + o) = make_float4(fmaf(dgi, u4.x, -a.x), fmaf(dgi, u4.y, -a.y), fmaf(dgi, u4.z, -a.z), fmaf(dgi, u4.w, -a.w));
  }
}

// Rare path (once per solve, one thread): iteration count, residual and status word.
__device__ __forceinline__ void write_stats(const CgParams& P, const double* red, int lp, int iter, int bad, double tol2) {
  double mx_all = 0.0;
#pragma unroll 1
  for (int c = 0; c < lp; ++c) mx_all = fmax(mx_all, red[2 * lp + c]);
  cg_write_stats(P, iter, sqrtf((float)mx_all), bad, mx_all, tol2);
}

template <bool SINGLE, bool TRACE>
__global__ void __launch_bounds__(CR_THREADS, 1) cg_resident_kernel(CrParams R) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const CgParams& P = R.cg;
  const int lp = P.lp, Q = lp >> 2, E3 = 3 * lp;
  const int G = gridDim.x, b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  const int row0 = min(P.m, b * R.rows_cap);
  const int rows = min(P.m, row0 + R.rows_cap) - row0;
  const size_t vec = (size_t)R.rows_cap * lp;

  // ---- shared memory carve-up (sizes mirrored by fixed_smem below) ----
  float* xs = reinterpret_cast<float*>(sm_raw);
  float* rs = xs + vec;
  float* ps = rs + vec;
  float* ss = ps + vec;
  float* ws = ss + vec;
  float* us = ws + vec;                           // SINGLE only: u = r/diag (otherwise u lives in global memory)
  float* dg = us + (SINGLE ? vec : 0);            // diag          [rows_cap]
  float* dinv = dg + R.rows_cap;                  // 1/diag        [rows_cap]
  int* rseg = reinterpret_cast<int*>(dinv + R.rows_cap);  // first segment of every row [rows_cap + 1]
  double* red = reinterpret_cast<double*>(sm_raw + align_up((size_t)((char*)(rseg + R.rows_cap + 1) - (char*)sm_raw), 16));  // [3*lp] g', d, rr
  float* inv_g_old = reinterpret_cast<float*>(red + E3);       // [lp]  1/<r,u> of the previous pass
  float* inv_a_old = inv_g_old + lp;                           // [lp]  1/alpha of the previous pass
  float* alpha = inv_a_old + lp;                               // [lp]
  float* beta = alpha + lp;                                    // [lp]
  int* frozen = reinterpret_cast<int*>(beta + lp);             // [lp]
  Ctrl* ctrl = reinterpret_cast<Ctrl*>(frozen + lp);           // 16 bytes
  float* spart = reinterpret_cast<float*>(reinterpret_cast<int*>(ctrl) + 4);  // [seg_cap][lp] segment sums (16-byte aligned)
  int* ecol = reinterpret_cast<int*>(spart + (size_t)R.seg_cap * lp);         // [seg_cap][CR_SEG] column (-1 = padding)
  float* eval = reinterpret_cast<float*>(ecol + (size_t)R.seg_cap * CR_SEG);  // [seg_cap][CR_SEG]

  // ---- segments: row i owns ceil(deg_i / CR_SEG) of them, numbered consecutively ----
  if (warp == 0) {
    const int per = (rows + 31) >> 5;
    const int lo = min(rows, lane * per), hi = min(rows, lo + per);
    int sum = 0;
#pragma unroll 1
    for (int i = lo; i < hi; ++i) sum += (__ldg(P.ptr + row0 + i + 1) - __ldg(P.ptr + row0 + i) + CR_SEG - 1) / CR_SEG;
    int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(FULL, incl, o);
      if (lane >= o) incl += t;
    }
    int run = incl - sum;
#pragma unroll 1
    for (int i = lo; i < hi; ++i) {
      rseg[i] = run;
      run += (__ldg(P.ptr + row0 + i + 1) - __ldg(P.ptr + row0 + i) + CR_SEG - 1) / CR_SEG;
    }
    if (lane == 31) rseg[rows] = incl;
  }
#pragma unroll 1
  for (int i = tid; i < rows; i += CR_THREADS) {
    const float d = __ldg(P.diag + row0 + i);
    dg[i] = d;
    dinv[i] = 1.f / d;
  }
#pragma unroll 1
  for (int c = tid; c < lp; c += CR_THREADS) {
    inv_g_old[c] = 1.f;
    inv_a_old[c] = 1.f;
    frozen[c] = 0;
  }
#pragma unroll 1
  for (int c = tid; c < E3; c += CR_THREADS) red[c] = 0.0;  // padded class columns stay zero
  __syncthreads();
  const int nseg = rseg[rows];
  const bool fits = nseg <= R.seg_cap;  // otherwise (huge row blocks) the SpMV walks the CSR in global memory row by row
  if (fits) {
#pragma unroll 1
    for (int i = warp; i < rows; i += CR_WARPS) {
      const int e0 = __ldg(P.ptr + row0 + i), deg = __ldg(P.ptr + row0 + i + 1) - e0;
      const int s0 = rseg[i] * CR_SEG, npad = (rseg[i + 1] - rseg[i]) * CR_SEG;
#pragma unroll 1
      for (int e = lane; e < npad; e += 32) {
        ecol[s0 + e] = (e < deg) ? __ldg(P.col + e0 + e) : -1;
        eval[s0 + e] = (e < deg) ? __ldg(P.val + e0 + e) : 0.f;
      }
    }
  }
  // Thread t works on class quad q = t mod Q of rows (or segments) t / Q, t / Q + istep, ...: the first Q * istep threads
  // are active and nothing inside the iteration divides by Q.
  const int istep = CR_THREADS / Q, q = tid % Q, i_first = (tid < istep * Q) ? tid / Q : (1 << 30);
  // x = 0, r = b, p = s = 0; publish u0 = r/diag
#pragma unroll 1
  for (int i = i_first; i < rows; i += istep) {
    const size_t o = (size_t)i * lp + 4 * q;
    const float4 bq = cg_load_rhs4(P, row0 + i, q);
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    *reinterpret_cast<float4*>(xs + o) = z;
    *reinterpret_cast<float4*>(rs + o) = bq;
    *reinterpret_cast<float4*>(ps + o) = z;
    *reinterpret_cast<float4*>(ss + o) = z;
    if (SINGLE)
      *reinterpret_cast<float4*>(us + o) = scale4(bq, dinv[i]);
    else
      *reinterpret_cast<float4*>(R.ubuf + (size_t)(row0 + i) * R.ustride + 4 * q) = scale4(bq, dinv[i]);
  }

  int iter = 0;
  unsigned nbar = 0;
  const float* ub = SINGLE ? us : R.ubuf;
  const int ust = SINGLE ? lp : R.ustride;
  const int jobs = 3 * P.l;  // (product, class column) pairs: <r,u>, <w,u>, <r,r>

  // The loop body is kept SMALL on purpose (~1 k instructions): the SM's instruction cache holds ~32 KB, a body that
  // does not fit is re-fetched from L2 every pass, and a phase executed by a single warp then pays the full fetch latency
  // per 128-byte line (measured: a 120-instruction scalar section took 3.9 us, profiles/r02_cg_trace.md).  Hence: no
  // single-warp phase, loops with warp-uniform trip counts (no divergent-shuffle slow paths), rare paths out of line.
  while (true) {
    // ================= (B) u of this pass is visible everywhere =================
    if (TRACE) cr_stamp(R, iter, 0);
    if (SINGLE) {
      __syncthreads();
    } else {
      nbar += (unsigned)G;
      grid_barrier(R.counter, nbar);
    }
    if (TRACE) cr_stamp(R, iter, 1);
    // ================= w = A u for my rows =================
    if (fits) {
#pragma unroll 1
      for (int sg = i_first; sg < nseg; sg += istep) {
        const int2* cp = reinterpret_cast<const int2*>(ecol + (size_t)sg * CR_SEG);   // CR_SEG is even: 8-byte aligned
        const float2* vp = reinterpret_cast<const float2*>(eval + (size_t)sg * CR_SEG);
        float4 u[CR_SEG];
#pragma unroll
        for (int e = 0; e < CR_SEG; e += 2) {
          const int2 cj = cp[e >> 1];
          u[e] = make_float4(0.f, 0.f, 0.f, 0.f);
          u[e + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (cj.x >= 0) u[e] = SINGLE ? *reinterpret_cast<const float4*>(ub + (size_t)cj.x * ust + 4 * q) : ldcg4(ub + (size_t)cj.x * ust + 4 * q);
          if (cj.y >= 0) u[e + 1] = SINGLE ? *reinterpret_cast<const float4*>(ub + (size_t)cj.y * ust + 4 * q) : ldcg4(ub + (size_t)cj.y * ust + 4 * q);
        }
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int e = 0; e < CR_SEG; e += 2) {  // the edge values are only read now, behind the gathers (registers)
          const float2 vj = vp[e >> 1];
          fma4(a, vj.x, u[e]);
          fma4(a, vj.y, u[e + 1]);
        }
        *reinterpret_cast<float4*>(spart + (size_t)sg * lp + 4 * q) = a;
      }
      if (TRACE) cr_stamp(R, iter, 2);
      __syncthreads();
      if (TRACE) cr_stamp(R, iter, 3);
#pragma unroll 1
      for (int i = i_first; i < rows; i += istep) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
        for (int sg = rseg[i]; sg < rseg[i + 1]; ++sg) {
          const float4 sp = *reinterpret_cast<const float4*>(spart + (size_t)sg * lp + 4 * q);
          a.x += sp.x; a.y += sp.y; a.z += sp.z; a.w += sp.w;
        }
        const size_t o = (size_t)i * lp + 4 * q;
        const float4 u4 = scale4(*reinterpret_cast<const float4*>(rs + o), dinv[i]);
        const float dgi = dg[i];
        *reinterpret_cast<float4*>(ws + o) = make_float4(fmaf(dgi, u4.x, -a.x), fmaf(dgi, u4.y, -a.y), fmaf(dgi, u4.z, -a.z), fmaf(dgi, u4.w, -a.w));
      }
    } else {
      spmv_rows_from_global<SINGLE>(P, row0, rows, ub, ust, rs, ws, dg, dinv);
    }
    if (TRACE) cr_stamp(R, iter, 4);
    __syncthreads();
    if (TRACE) cr_stamp(R, iter, 5);
    // ================= partial <r,u>, <w,u>, <r,r>: one warp per (product, class column), one butterfly each =========
    if (tid == 0) ctrl->flags = 0;  // read last before the previous pass's vector update; set again after barrier (A)
#pragma unroll 1
    for (int job = warp; job < jobs; job += CR_WARPS) {
      const int v = (job >= 2 * P.l) ? 2 : (job >= P.l ? 1 : 0), cc = job - v * P.l;
      const float* av = (v == 1) ? ws : rs;
      double t = 0.0;
#pragma unroll 4
      for (int i0 = 0; i0 < rows; i0 += 32) {  // warp-uniform trip count; unrolled: the shared-memory loads go out together
        const int i = i0 + lane;
        if (i < rows) {
          const float r = rs[(size_t)i * lp + cc];
          t += (double)av[(size_t)i * lp + cc] * (double)((v == 2) ? r : r * dinv[i]);
        }
      }
      t = warp_sum(t);  // xor butterfly: fixed order
      if (lane == 0) {
        if (SINGLE)
          red[v * lp + cc] = t;
        else
          R.part[(size_t)(v * lp + cc) * G + b] = t;  // column-major: the readers' loads are coalesced
      }
    }
    if (TRACE) cr_stamp(R, iter, 6);
    // ================= (A) dot products over all CTAs =================
    if (SINGLE) {
      __syncthreads();
    } else {
      nbar += (unsigned)G;
      grid_barrier(R.counter, nbar);
      if (TRACE) cr_stamp(R, iter, 7);
      // every CTA adds the G partials of every column itself, in the same order: one warp per column, all loads of a lane
      // in flight at once, one butterfly
#pragma unroll 1
      for (int job = warp; job < jobs; job += CR_WARPS) {
        const int v = (job >= 2 * P.l) ? 2 : (job >= P.l ? 1 : 0), e = v * lp + (job - v * P.l);
        const double* src = R.part + (size_t)e * G;
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < CR_MAX_GRID / 32; ++k)
          if (lane + 32 * k < G) t += __ldcg(src + lane + 32 * k);
        t = warp_sum(t);
        if (lane == 0) red[e] = t;
      }
      if (TRACE) cr_stamp(R, iter, 8);
      __syncthreads();
    }
    if (TRACE) cr_stamp(R, iter, 11);

    // ================= scalars: thread c owns class column c (every CTA computes identical values) =================
    if (iter == 0) {  // P.tol < 0: relative to the largest right-hand-side column norm (r = b at this point)
      if (tid == 0) {
        double mx = 0.0;
#pragma unroll 1
        for (int c = 0; c < lp; ++c) mx = fmax(mx, red[2 * lp + c]);
        ctrl->tol2 = (P.tol < 0.f) ? (double)P.tol * (double)P.tol * mx : (double)P.tol * (double)P.tol;
      }
      __syncthreads();
    }
    int live = 0, bad = 0;
    if (tid < lp) {
      const int c = tid;
      const double tol2 = ctrl->tol2;
      const double g_new = red[c], d_new = red[lp + c], rr = red[2 * lp + c];
      bad = (!(rr == rr) || rr > 1.0e300) ? 1 : 0;
      float al = 0.f, be = 0.f;
      if (!frozen[c] && rr > tol2) {  // columns that broke down are frozen for good
        live = 1;
        cg_column_step(g_new, d_new, iter == 0, inv_g_old[c], inv_a_old[c], frozen[c], al, be);
      }
      alpha[c] = al;
      beta[c] = be;
    }
    if (live | bad) atomicOr(&ctrl->flags, live | (bad << 1));
    __syncthreads();
    const int any_live = ctrl->flags & 1, any_bad = ctrl->flags & 2;
    if (TRACE) cr_stamp(R, iter, 14);
    if (any_bad || !any_live || iter >= P.max_iter) {
      if (b == 0 && tid == 0) write_stats(P, red, lp, iter, any_bad, ctrl->tol2);
      if (!SINGLE && P.ext_counter != nullptr && tid == 0) {
        // exit ticket: every CTA is past its last barrier wait when it gets here, so the last one may rewind both words
        if (atomicAdd(P.ext_counter + 1, 1u) == (unsigned)G - 1u) {
          P.ext_counter[0] = 0u;
          P.ext_counter[1] = 0u;
        }
      }
      break;
    }
    ++iter;
    // ================= vector updates (all on chip), publish the new u =================
#pragma unroll 1
    for (int i = i_first; i < rows; i += istep) {
      const size_t o = (size_t)i * lp + 4 * q;
      const float4 al = *reinterpret_cast<const float4*>(alpha + 4 * q);
      const float4 be = *reinterpret_cast<const float4*>(beta + 4 * q);
      const float di = dinv[i];
      float4 x4 = *reinterpret_cast<const float4*>(xs + o), r4 = *reinterpret_cast<const float4*>(rs + o);
      float4 p4 = *reinterpret_cast<const float4*>(ps + o), s4 = *reinterpret_cast<const float4*>(ss + o);
      const float4 w4 = *reinterpret_cast<const float4*>(ws + o);
      cg_cg_update(al, be, scale4(r4, di), w4, x4, r4, p4, s4);
      *reinterpret_cast<float4*>(xs + o) = x4;
      *reinterpret_cast<float4*>(rs + o) = r4;
      *reinterpret_cast<float4*>(ps + o) = p4;
      *reinterpret_cast<float4*>(ss + o) = s4;
      if (SINGLE)
        *reinterpret_cast<float4*>(us + o) = scale4(r4, di);
      else
        *reinterpret_cast<float4*>(R.ubuf + (size_t)(row0 + i) * R.ustride + 4 * q) = scale4(r4, di);
    }
    if (TRACE) cr_stamp(R, iter - 1, 15);
  }

  // ---- write the answer ----
#pragma unroll 1
  for (int i = i_first; i < rows; i += istep) {
    const float4 x4 = *reinterpret_cast<const float4*>(xs + (size_t)i * lp + 4 * q);
    *reinterpret_cast<float4*>(P.x + (size_t)(row0 + i) * lp + 4 * q) = x4;
    cg_store_copy4(P, row0 + i, q, x4);
  }
}

size_t fixed_smem(int rows_cap, int lp, bool single) {
  const int E3 = 3 * lp;
  size_t b = sizeof(float) * ((single ? 6 : 5) * (size_t)rows_cap * lp + 2 * (size_t)rows_cap) + sizeof(int) * ((size_t)rows_cap + 1);
  b = align_up(b, 16);
  b += sizeof(double) * (size_t)E3 + sizeof(float) * (4 * (size_t)lp) + sizeof(int) * lp + 16;
  return align_up(b, 16);
}

int ustride_of(int lp) { return lp <= 4 ? 4 : (lp <= 8 ? 8 : (lp <= 16 ? 16 : lp)); }

struct CrPlan {
  int ok, grid, rows_cap, seg_cap;
  size_t smem;
};

CrPlan plan(int m, int lp) {
  CrPlan p;
  p.ok = 0;
  const int sms = device_info().sms;
  const size_t per_seg = align_up(sizeof(int) * CR_SEG + sizeof(float) * CR_SEG + sizeof(float) * lp, 16);
  int grid;
  // whole system in one SM (no grid-wide exchange at all) when the vectors and ~5 segments per row fit
  if (fixed_smem(m, lp, true) + per_seg * 5 * (size_t)m <= CR_SMEM_BUDGET * 3 / 4)
    grid = 1;
  else
    grid = max(2, min(min(sms, CR_MAX_GRID), ceil_div(m, 96)));
  int rows_cap = ceil_div(m, grid);
  if (grid > 1 && fixed_smem(rows_cap, lp, false) + 4 * 1024 > CR_SMEM_BUDGET) {
    grid = min(sms, CR_MAX_GRID);
    rows_cap = ceil_div(m, grid);
    if (fixed_smem(rows_cap, lp, false) + 4 * 1024 > CR_SMEM_BUDGET) return p;  // does not fit on chip: streaming kernel
  }
  p.grid = grid;
  p.rows_cap = rows_cap;
  const size_t fx = fixed_smem(rows_cap, lp, grid == 1);
  p.seg_cap = (int)((CR_SMEM_BUDGET - fx) / per_seg);
  p.smem = fx + (size_t)p.seg_cap * per_seg;
  p.ok = 1;
  return p;
}

}  // namespace

static unsigned long long* g_cg_trace = nullptr;
void cg_set_trace(void* buf) { g_cg_trace = (unsigned long long*)buf; }
void* cg_get_trace() { return g_cg_trace; }

size_t cg_resident_ws_bytes(int m, int lp) {
  const size_t sms = (size_t)device_info().sms;
  return align_up(sizeof(float) * (size_t)m * ustride_of(lp), 256) + align_up(sizeof(double) * 3 * (size_t)lp * sms, 256) + 256 + 256;
}

bool cg_resident_fits(int m, int lp) { return plan(m, lp).ok != 0; }

int cg_resident_launch(const CgParams& P, void* scratch, cudaStream_t st) {
  const CrPlan pl = plan(P.m, P.lp);
  CrParams R;
  R.cg = P;
  Carver cv(scratch, cg_resident_ws_bytes(P.m, P.lp));
  const size_t sms = (size_t)device_info().sms;
  R.ustride = ustride_of(P.lp);
  R.ubuf = cv.take<float>((size_t)P.m * R.ustride);
  R.part = cv.take<double>(3 * (size_t)P.lp * sms);
  R.counter = cv.take<unsigned>(64);
  if (P.ext_counter != nullptr) R.counter = P.ext_counter;
  R.rows_cap = pl.rows_cap;
  R.seg_cap = pl.seg_cap;
  R.trace = g_cg_trace;
  const void* k_single = (const void*)cg_resident_kernel<true, false>;
  const void* k_multi = (const void*)cg_resident_kernel<false, false>;
  if (R.trace != nullptr) k_multi = (const void*)cg_resident_kernel<false, true>;  // debug timeline (gll_debug_cg_trace)
  GLL_CUDA_CHECK(set_max_dynamic_smem_once(k_single, (int)CR_SMEM_BUDGET));
  GLL_CUDA_CHECK(set_max_dynamic_smem_once(k_multi, (int)CR_SMEM_BUDGET));
  void* args[] = {&R};
  if (pl.grid == 1) {
    GLL_PROF(KID_CG, st);
    GLL_CUDA_CHECK(cudaLaunchKernel(k_single, dim3(1), dim3(CR_THREADS), args, pl.smem, st));
  } else {
    // only the barrier counter needs a defined start value (the partials of padded class columns are never read)
    if (P.ext_counter == nullptr) GLL_CUDA_CHECK(cudaMemsetAsync(R.counter, 0, 64 * sizeof(unsigned), st));
    GLL_PROF(KID_CG, st);
    // cooperative launch: all CTAs are co-resident, which the grid barrier relies on
    GLL_CUDA_CHECK(cudaLaunchCooperativeKernel(k_multi, dim3(pl.grid), dim3(CR_THREADS), args, pl.smem, st));
  }
  return GLL_OK;
}

}  // namespace gll
