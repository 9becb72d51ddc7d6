// K4, row-partitioned: the CG solve of ONE graph spread over R ranks by row blocks (SURVEY 8e, the north star's first
// variant): rank r owns rows [row_lo, row_hi) of x, r, p, s; per iteration the host exchanges the iterate with one NCCL
// all-gather and the dot products with one NCCL all-reduce.  Same arithmetic as cg_resident.cu: Jacobi-preconditioned
// Chronopoulos-Gear CG (one SpMV and ONE fused reduction per iteration), per-column freeze and stop test of
// stable_conjgrad (GLL.py:247-276).
//
//   init     x = 0, r = b, u = r / diag (own rows of the shared u array), p = s = 0
//   loop     [all-gather u]                                                  <- host, NCCL
//            spmv    w = A u (own rows), sums = {<r,u>, <w,u>, <r,r>} over own rows (fp64, fixed summation order)
//            [all-reduce sums]                                               <- host, NCCL
//            update  beta = g/g_old, alpha = g/(d - beta g/alpha_old); p = u + beta p; s = w + beta s; x += alpha p;
//                    r -= alpha s; u = r/diag     (every CTA derives the same scalars from the same reduced sums)
//
// No floating-point atomics: per-CTA partials -> the last CTA to finish (integer ticket) adds them in CTA order.
//
// Peer-memory mode (gll_cg_rows_*_p2p): the two collectives are FUSED into the kernels over NVLink peer pointers
// (symmetric memory) -- no NCCL call, no host round trip inside the loop:
//   update / init   store the new u rows straight into EVERY rank's copy of the u array (P2P stores), then the last CTA
//                   raises this rank's "u published" epoch flag on every peer (fence.sys, st.release.sys)
//   spmv            waits (ld.acquire.sys on LOCAL flags, bounded spin) until every rank's u for this iteration has
//                   landed; its last CTA writes this rank's 3*lp partial sums into a mailbox row on every peer and raises
//                   the "sums published" flag
//   update          waits for all ranks' sums, adds the mailbox rows in rank order (identical on every rank), proceeds
// Every wait is for data produced by kernels that the peers launch EARLIER in the same sequence, so the scheme cannot
// deadlock as long as every rank enqueues the same launches; a spin that lasts longer than 2 s traps (no hung GPU).
#include <stdlib.h>
#include <string.h>

#include "cg_common.cuh"

namespace gll {
namespace {

constexpr int RW_THREADS = 512;
constexpr int RW_WARPS = RW_THREADS / 32;

struct RowsState {
  float *r, *p, *s, *w;      // [rows_local][lp]
  double* partial;           // [grid][3*lp]
  unsigned* ticket;          // spmv: last-CTA election
  unsigned* ticket2;         // init / update: last-CTA election for the "u published" flag (peer-memory mode)
  float* scal;               // [2 parities][3][lp]: 1/gamma_old, 1/alpha_old, frozen (0/1); launch `iter` reads parity
                             // iter&1 and CTA 0 writes the other one, so every CTA of a launch sees the same values
  double* tol2;              // resolved at iteration 0
  int grid;
};

int rows_grid() { return device_info().sms * 2; }

RowsState carve(void* ws, size_t ws_bytes, int rows_local, int lp) {
  Carver cv(ws, ws_bytes);
  RowsState S;
  const size_t v = (size_t)rows_local * lp;
  S.r = cv.take<float>(v);
  S.p = cv.take<float>(v);
  S.s = cv.take<float>(v);
  S.w = cv.take<float>(v);
  S.grid = rows_grid();
  S.partial = cv.take<double>((size_t)S.grid * 3 * lp);
  S.ticket = cv.take<unsigned>(64);
  S.ticket2 = S.ticket + 32;
  S.scal = cv.take<float>(6 * (size_t)lp);
  S.tol2 = cv.take<double>(4);
  return S;
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }

// ---- peer-memory mode ----
constexpr int MAX_PEERS = 8;
constexpr int MAIL_ROW = 3 * CG_MAX_LP;  // doubles per (parity, source rank)
struct Peers {
  float* u[MAX_PEERS];      // every rank's u array (m' x lp), mine included
  double* mail[MAX_PEERS];  // every rank's mailbox: [2 parities][MAX_PEERS sources][MAIL_ROW]
  unsigned* flags[MAX_PEERS];  // every rank's flags: [0][src] = epoch of src's published u, [1][src] = of src's sums
  int world, rank;          // world == 0: not in peer-memory mode
  unsigned long long timeout_ns;  // bound of a flag wait (GLL_B200_PEER_TIMEOUT_S, default 60 s)
};
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// one thread: until every rank's flag has reached `epoch` (flags only grow).  The wait is bounded so that a dead peer or
// diverged launch sequences end in an error instead of a hung GPU; the bound is long (a peer's HOST may stall for seconds:
// lazy module loading on its first call, garbage collection, a debugger) and configurable.
__device__ __forceinline__ void wait_all_flags(const unsigned* f, int world, unsigned epoch, unsigned long long timeout_ns) {
  unsigned long long t0, t1;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (int p = 0; p < world; ++p) {
    unsigned spin = 0;
    while ((int)(ld_acquire_sys(f + p) - epoch) < 0) {
      if ((++spin & 1023u) == 0) {
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > timeout_ns) __trap();  // a peer died or the launch sequences diverged
      }
    }
  }
}
// whole CTA, at the end of a kernel whose threads stored into peer memory: the last CTA to get here raises flag `which`
__device__ __forceinline__ void publish_epoch(const Peers& P, int which, unsigned epoch, unsigned* ticket) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();  // this CTA's peer stores (ordered before me by the barrier) are performed system-wide
    if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
      __threadfence_system();
      *ticket = 0u;
      for (int p = 0; p < P.world; ++p) st_release_sys(P.flags[p] + which * MAX_PEERS + P.rank, epoch);
    }
  }
}

__global__ void __launch_bounds__(256)
rows_init_kernel(const float* __restrict__ diag, const float* __restrict__ rhs, int lp, int row_lo, int row_hi, float* __restrict__ x,
                 float* __restrict__ u_full, RowsState S, Peers PR, unsigned epoch) {
  const int Q = lp >> 2;
  const long long total = (long long)(row_hi - row_lo) * Q;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int li = (int)(t / Q), q = (int)(t - (long long)li * Q);
    const int i = row_lo + li;
    const float4 b = ld4(rhs + (size_t)i * lp + 4 * q);
    const float dinv = 1.f / __ldg(diag + i);
    const size_t lo = (size_t)li * lp + 4 * q;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    st4(x + (size_t)i * lp + 4 * q, z);
    st4(S.r + lo, b);
    st4(S.p + lo, z);
    st4(S.s + lo, z);
    const float4 u4 = make_float4(b.x * dinv, b.y * dinv, b.z * dinv, b.w * dinv);
    if (PR.world == 0) {
      st4(u_full + (size_t)i * lp + 4 * q, u4);
    } else {
      for (int p = 0; p < PR.world; ++p) st4(PR.u[p] + (size_t)i * lp + 4 * q, u4);
    }
  }
  if (blockIdx.x == 0) {
    for (int c = threadIdx.x; c < 6 * lp; c += blockDim.x) S.scal[c] = 0.f;
    if (threadIdx.x == 0) {
      *S.ticket = 0u;
      *S.tol2 = 0.0;
    }
  }
  if (PR.world > 0) publish_epoch(PR, 0, epoch, S.ticket2);
}

// w = A u on the rank's rows; lane = (neighbour slot s, class quad q), 128-bit gathers of u_j, four gathers in flight
__global__ void __launch_bounds__(RW_THREADS)
rows_spmv_kernel(const int* __restrict__ ptr, const int* __restrict__ col, const float* __restrict__ val, const float* __restrict__ diag,
                 int lp, int row_lo, int row_hi, const float* __restrict__ u_full, RowsState S, double* __restrict__ sums, Peers PR,
                 unsigned epoch, const int* __restrict__ ctrl) {
  extern __shared__ double wpart[];  // [RW_WARPS][3*lp]
  __shared__ bool last;
  if (PR.world > 0) {
    if (ctrl[0] != 0) return;  // the solve has stopped on every rank (same decision everywhere): nothing to wait for
    if (threadIdx.x == 0) wait_all_flags(PR.flags[PR.rank], PR.world, epoch, PR.timeout_ns);  // everybody's u of this iteration is here
    __syncthreads();
  }
  const int Q = lp >> 2, NS = 32 / Q;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int s = lane / Q, q = lane - s * Q;
  const bool active = lane < NS * Q;
  double g[4] = {0, 0, 0, 0}, dd[4] = {0, 0, 0, 0}, rr[4] = {0, 0, 0, 0};
  for (int i = row_lo + blockIdx.x * RW_WARPS + warp; i < row_hi; i += gridDim.x * RW_WARPS) {
    const int e0 = __ldg(ptr + i), e1 = __ldg(ptr + i + 1);
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    if (active) {
      for (int e = e0 + s; e < e1; e += 4 * NS) {
        float wv[4];
        float4 uj[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int et = e + t * NS;
          const bool ok = et < e1;
          const int j = ok ? __ldg(col + et) : i;
          wv[t] = ok ? __ldg(val + et) : 0.f;
          uj[t] = ld4(u_full + (size_t)j * lp + 4 * q);
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          a.x = fmaf(wv[t], uj[t].x, a.x);
          a.y = fmaf(wv[t], uj[t].y, a.y);
          a.z = fmaf(wv[t], uj[t].z, a.z);
          a.w = fmaf(wv[t], uj[t].w, a.w);
        }
      }
    }
    a = reduce_over_s(a, s, NS, Q);
    if (lane < Q) {
      const size_t lo = (size_t)(i - row_lo) * lp + 4 * lane;
      const float4 ui = ld4(u_full + (size_t)i * lp + 4 * lane);
      const float4 ri = ld4(S.r + lo);
      const float dg = __ldg(diag + i);
      const float4 w = make_float4(fmaf(dg, ui.x, -a.x), fmaf(dg, ui.y, -a.y), fmaf(dg, ui.z, -a.z), fmaf(dg, ui.w, -a.w));
      st4(S.w + lo, w);
      g[0] += (double)ri.x * ui.x; g[1] += (double)ri.y * ui.y; g[2] += (double)ri.z * ui.z; g[3] += (double)ri.w * ui.w;
      dd[0] += (double)w.x * ui.x; dd[1] += (double)w.y * ui.y; dd[2] += (double)w.z * ui.z; dd[3] += (double)w.w * ui.w;
      rr[0] += (double)ri.x * ri.x; rr[1] += (double)ri.y * ri.y; rr[2] += (double)ri.z * ri.z; rr[3] += (double)ri.w * ri.w;
    }
  }
  if (lane < Q) {
    double* d = wpart + (size_t)warp * 3 * lp;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      d[4 * lane + t] = g[t];
      d[lp + 4 * lane + t] = dd[t];
      d[2 * lp + 4 * lane + t] = rr[t];
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 3 * lp; c += RW_THREADS) {
    double t = 0.0;
    for (int w = 0; w < RW_WARPS; ++w) t += wpart[(size_t)w * 3 * lp + c];
    S.partial[(size_t)blockIdx.x * 3 * lp + c] = t;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = (atomicAdd(S.ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!last) return;
  __threadfence();
  for (int c = threadIdx.x; c < 3 * lp; c += RW_THREADS) {
    double t = 0.0;
    for (int b = 0; b < (int)gridDim.x; ++b) t += __ldcg(S.partial + (size_t)b * 3 * lp + c);
    if (PR.world == 0) {
      sums[c] = t;
    } else {  // my partial sums into my mailbox row on every rank
      for (int p = 0; p < PR.world; ++p) PR.mail[p][((size_t)(epoch & 1u) * MAX_PEERS + PR.rank) * MAIL_ROW + c] = t;
    }
  }
  if (PR.world > 0) {
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0)
      for (int p = 0; p < PR.world; ++p) st_release_sys(PR.flags[p] + MAX_PEERS + PR.rank, epoch);
  }
  if (threadIdx.x == 0) *S.ticket = 0u;
}

// ctrl[0] = stop flag, ctrl[1] = iterations done, ctrl[2] = status bits
__global__ void __launch_bounds__(256)
rows_update_kernel(const float* __restrict__ diag, int lp, int row_lo, int row_hi, const double* sums, int iter,
                   int max_iter, float tol, float* __restrict__ x, float* __restrict__ u_full, RowsState S, int* __restrict__ ctrl,
                   float* __restrict__ resid_out, Peers PR, unsigned epoch) {
  __shared__ float alpha[CG_MAX_LP], beta[CG_MAX_LP];
  __shared__ double ssum[MAIL_ROW];
  __shared__ int stop_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float* sc_old = S.scal + (size_t)(iter & 1) * 3 * lp;
  float* sc_new = S.scal + (size_t)((iter + 1) & 1) * 3 * lp;
  if (ctrl[0] != 0) return;  // an earlier launch stopped the solve (written by that launch, so no race here)
  if (PR.world > 0) {  // every rank's partial sums of this iteration: add the mailbox rows in rank order
    if (threadIdx.x == 0) wait_all_flags(PR.flags[PR.rank] + MAX_PEERS, PR.world, epoch, PR.timeout_ns);
    __syncthreads();
    const double* mb = PR.mail[PR.rank] + (size_t)(epoch & 1u) * MAX_PEERS * MAIL_ROW;
    for (int c = threadIdx.x; c < 3 * lp; c += blockDim.x) {
      double t = 0.0;
      for (int p = 0; p < PR.world; ++p) t += __ldcg(mb + (size_t)p * MAIL_ROW + c);
      ssum[c] = t;
    }
    __syncthreads();
    sums = ssum;
  }
  if (warp == 0) {
    double tol2;
    if (iter == 0) {
      double mx = 0.0;
      for (int c = lane; c < lp; c += 32) mx = fmax(mx, sums[2 * lp + c]);
      for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(FULL, mx, o));
      tol2 = (tol < 0.f) ? (double)tol * (double)tol * mx : (double)tol * (double)tol;
    } else {
      tol2 = *S.tol2;
    }
    double mx_all = 0.0, mx_live = 0.0;
    int bad = 0;
    for (int c = lane; c < lp; c += 32) {
      const double v = sums[2 * lp + c];
      bad |= (!(v == v) || v > 1.0e300) ? 1 : 0;
      mx_all = fmax(mx_all, v);
      if (sc_old[2 * lp + c] == 0.f) mx_live = fmax(mx_live, v);
    }
    for (int o = 16; o > 0; o >>= 1) {
      mx_all = fmax(mx_all, __shfl_xor_sync(FULL, mx_all, o));
      mx_live = fmax(mx_live, __shfl_xor_sync(FULL, mx_live, o));
      bad |= __shfl_xor_sync(FULL, bad, o);
    }
    const bool stop = bad || mx_live <= tol2 || iter >= max_iter;
    if (lane == 0) stop_s = stop ? 1 : 0;
    if (blockIdx.x == 0) {
      if (lane == 0) {
        if (iter == 0) *S.tol2 = tol2;
        if (stop) {
          ctrl[0] = 1;
          ctrl[1] = iter;
          int st = 0;
          if (bad) st |= GLL_STATUS_NONFINITE;
          if (!bad && !(mx_all <= tol2)) st |= GLL_STATUS_CG_NOT_CONVERGED;
          ctrl[2] |= st;
          if (resid_out) *resid_out = sqrtf((float)mx_all);
        }
      }
    }
    for (int c = lane; c < lp; c += 32) {
      const double g_new = sums[c], d_new = sums[lp + c], rr = sums[2 * lp + c];
      float al = 0.f, be = 0.f, ig = sc_old[c], ia = sc_old[lp + c];
      int fr = sc_old[2 * lp + c] != 0.f;
      if (!stop && !fr && rr > tol2) {
        const float bb = (iter == 0) ? 0.f : (float)g_new * ig;
        const double den = d_new - (double)bb * g_new * (double)ia;
        if (den > 0.0 && g_new > 0.0) {
          al = (float)g_new / (float)den;
          be = bb;
          ia = 1.f / al;
          ig = 1.f / (float)g_new;
        } else {
          fr = 1;  // breakdown at the fp32 floor: stop moving this column
        }
      }
      alpha[c] = al;
      beta[c] = be;
      if (blockIdx.x == 0) {
        sc_new[c] = ig;
        sc_new[lp + c] = ia;
        sc_new[2 * lp + c] = fr ? 1.f : 0.f;
      }
    }
  }
  __syncthreads();
  if (stop_s) return;
  const int Q = lp >> 2;
  const long long total = (long long)(row_hi - row_lo) * Q;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int li = (int)(t / Q), q = (int)(t - (long long)li * Q);
    const int i = row_lo + li;
    const size_t lo = (size_t)li * lp + 4 * q, go = (size_t)i * lp + 4 * q;
    const float4 al = ld4(alpha + 4 * q), be = ld4(beta + 4 * q);
    const float4 u = ld4(u_full + go), w = ld4(S.w + lo);
    float4 p = ld4(S.p + lo), sv = ld4(S.s + lo), xv = ld4(x + go), r = ld4(S.r + lo);
    cg_cg_update(al, be, u, w, xv, r, p, sv);
    const float dinv = 1.f / __ldg(diag + i);
    st4(S.p + lo, p);
    st4(S.s + lo, sv);
    st4(x + go, xv);
    st4(S.r + lo, r);
    const float4 un = make_float4(r.x * dinv, r.y * dinv, r.z * dinv, r.w * dinv);
    if (PR.world == 0) {
      st4(u_full + go, un);
    } else {  // the fused all-gather: my rows of the new u into every rank's copy
      for (int p = 0; p < PR.world; ++p) st4(PR.u[p] + go, un);
    }
  }
  if (PR.world > 0) publish_epoch(PR, 0, epoch + 1u, S.ticket2);
}

}  // namespace

size_t cg_rows_ws_bytes(int rows_local, int l) {
  const int lp = padded_classes(l);
  const size_t v = align_up(sizeof(float) * (size_t)rows_local * lp, 256);
  return 4 * v + align_up(sizeof(double) * (size_t)rows_grid() * 3 * lp, 256) + 256 + align_up(sizeof(float) * 6 * lp, 256) + 256 + 2048;
}

static Peers make_peers(const gll_peers* pr) {
  Peers P;
  memset(&P, 0, sizeof(P));
  if (pr != nullptr) {
    static const double timeout_s = [] {
      const char* e = getenv("GLL_B200_PEER_TIMEOUT_S");
      const double v = e ? atof(e) : 0.0;
      return v > 0.0 ? v : 60.0;
    }();
    P.timeout_ns = (unsigned long long)(timeout_s * 1e9);
    P.world = pr->world;
    P.rank = pr->rank;
    for (int p = 0; p < pr->world && p < MAX_PEERS; ++p) {
      P.u[p] = (float*)pr->u[p];
      P.mail[p] = (double*)pr->mail[p];
      P.flags[p] = (unsigned*)pr->flags[p];
    }
  }
  return P;
}
static bool peers_ok(const gll_peers* pr) {
  if (pr == nullptr) return true;
  if (pr->world < 1 || pr->world > MAX_PEERS || pr->rank < 0 || pr->rank >= pr->world) return false;
  for (int p = 0; p < pr->world; ++p)
    if (!pr->u[p] || !pr->mail[p] || !pr->flags[p]) return false;
  return true;
}
size_t cg_rows_peer_mail_bytes() { return sizeof(double) * 2 * MAX_PEERS * MAIL_ROW; }
size_t cg_rows_peer_flag_bytes() { return sizeof(unsigned) * 2 * MAX_PEERS; }

int cg_rows_init(const float* diag, const float* rhs, int m, int l, int row_lo, int row_hi, float* x, float* u_full, void* ws,
                 size_t ws_bytes, const gll_peers* peers, unsigned epoch, cudaStream_t st) {
  GLL_REQUIRE(peers_ok(peers), "bad peer table");
  GLL_REQUIRE(diag && rhs && x && u_full && ws, "null pointer");
  GLL_REQUIRE(m >= 1 && l >= 1 && 0 <= row_lo && row_lo <= row_hi && row_hi <= m, "bad sizes");
  const int lp = padded_classes(l);
  GLL_REQUIRE(lp <= CG_MAX_LP, "at most 128 classes per solve");
  if (ws_bytes < cg_rows_ws_bytes(row_hi - row_lo, l)) {
    set_error("row-partitioned CG workspace too small: %zu < %zu", ws_bytes, cg_rows_ws_bytes(row_hi - row_lo, l));
    return GLL_ERR_WORKSPACE;
  }
  RowsState S = carve(ws, ws_bytes, row_hi - row_lo, lp);
  const long long total = (long long)(row_hi - row_lo) * (lp >> 2);
  const int grid = (int)max(1LL, min((long long)device_info().sms * 8, (total + 255) / 256));
  GLL_CUDA_CHECK(cudaMemsetAsync(S.ticket, 0, 64 * sizeof(unsigned), st));  // both last-CTA tickets start at zero
  GLL_PROF(KID_CG_ROWS, st);
  rows_init_kernel<<<grid, 256, 0, st>>>(diag, rhs, lp, row_lo, row_hi, x, u_full, S, make_peers(peers), epoch);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

int cg_rows_spmv(const int* uu_ptr, const int* uu_col, const float* uu_val, const float* diag, int m, int l, int row_lo, int row_hi,
                 const float* u_full, double* sums, void* ws, size_t ws_bytes, const gll_peers* peers, unsigned epoch,
                 const int* ctrl, cudaStream_t st) {
  GLL_REQUIRE(uu_ptr && uu_col && uu_val && diag && u_full && ws && (sums || peers), "null pointer");
  GLL_REQUIRE(peers_ok(peers) && (peers == nullptr || ctrl != nullptr), "bad peer table");
  GLL_REQUIRE(m >= 1 && l >= 1 && 0 <= row_lo && row_lo <= row_hi && row_hi <= m, "bad sizes");
  const int lp = padded_classes(l);
  GLL_REQUIRE(lp <= CG_MAX_LP, "at most 128 classes per solve");
  RowsState S = carve(ws, ws_bytes, row_hi - row_lo, lp);
  const size_t smem = sizeof(double) * RW_WARPS * 3 * (size_t)lp;
  GLL_CUDA_CHECK(set_max_dynamic_smem_once((const void*)rows_spmv_kernel, (int)(sizeof(double) * RW_WARPS * 3 * CG_MAX_LP)));
  GLL_PROF(KID_CG_ROWS, st);
  rows_spmv_kernel<<<S.grid, RW_THREADS, smem, st>>>(uu_ptr, uu_col, uu_val, diag, lp, row_lo, row_hi, u_full, S, sums,
                                                     make_peers(peers), epoch, ctrl);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

int cg_rows_update(const float* diag, int m, int l, int row_lo, int row_hi, const double* sums, int iter, int max_iter, float tol,
                   float* x, float* u_full, int* ctrl, float* resid_out, void* ws, size_t ws_bytes, const gll_peers* peers,
                   unsigned epoch, cudaStream_t st) {
  GLL_REQUIRE(diag && (sums || peers) && x && u_full && ctrl && ws, "null pointer");
  GLL_REQUIRE(peers_ok(peers), "bad peer table");
  GLL_REQUIRE(m >= 1 && l >= 1 && 0 <= row_lo && row_lo <= row_hi && row_hi <= m && iter >= 0, "bad sizes");
  const int lp = padded_classes(l);
  RowsState S = carve(ws, ws_bytes, row_hi - row_lo, lp);
  const long long total = (long long)(row_hi - row_lo) * (lp >> 2);
  const int grid = (int)max(1LL, min((long long)device_info().sms * 8, (total + 255) / 256));
  GLL_PROF(KID_CG_ROWS, st);
  rows_update_kernel<<<grid, 256, 0, st>>>(diag, lp, row_lo, row_hi, sums, iter, max_iter, tol, x, u_full, S, ctrl, resid_out,
                                           make_peers(peers), epoch);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

}  // namespace gll
