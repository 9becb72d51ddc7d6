// K1 -- exact k-nearest-neighbour search (replaces gl.weightmatrix.knnsearch(..., 'annoy'), GLL.py:181-189).
//
// Pipeline (all on one stream, no host sync):
//   sqnorm      : ||x_i||^2 (fp64 accumulate -> fp32) and the global max; for the tensor-core path also the 16-bit operand
//                 split of X (fp16 hi/lo of the power-of-two scaled rows and the measured residual rho, or bf16 hi/lo)
//   gemm_topk   : tiled Gram GEMM  d~^2_ij = |x_i|^2 + |x_j|^2 - 2 x_i.x_j  with a FUSED per-row top-KC epilogue:
//                 a tile's distances are filtered against the row's running threshold and only the survivors
//                 touch shared memory; the n x n matrix never reaches HBM.  Column range split across CTAs.
//   rerank      : merge the per-split candidate lists, recompute the KC survivors as sum (x_i-x_j)^2 in fp64
//                 (bit-symmetric in i,j), order by (distance, index), emit k entries with self in slot 0, and
//                 PROVE completeness: every non-candidate has approximate distance >= L_i, so its true distance
//                 is >= L_i - err; rows where that does not exceed the k-th exact distance are queued for
//   fallback    : brute-force fp64 search for the queued rows only.
//
// This file holds the fp32 SIMT Gram path (tiny graphs; any d, any alignment), the operand-split kernels, re-rank and
// fallback, and the host code of every search.  The tcgen05/TMA Gram path (n >= 256, any d: rows are zero-padded to a multiple
// of 32) lives in knn_tc.cu; both paths end in the same re-rank and fallback (knn_finish).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include <cuda_fp16.h>

#include "common.cuh"
#include "knn_common.cuh"

namespace gll {
namespace {

constexpr int BM = 128, BN = 128, BK = 16, PAD = 4;
constexpr int GEMM_THREADS = 256;
constexpr int LDS_A = BM + PAD, LDS_B = BN + PAD;

constexpr size_t gemm_smem_bytes() {
  return sizeof(float) * (2 * BK * LDS_A + 2 * BK * LDS_B) + sizeof(u64) * (BM * KC + BM * BN) +
         sizeof(float) * BM + sizeof(int) * BM;
}

// Running maximum in one global word.  Every row contributes, and same-address atomics serialise in L2 (four per row cost
// more than the rest of the split kernel), so the atomic is only issued when the value read from L2 is still smaller: a
// stale read merely issues a redundant atomic, the maximum itself stays exact.
__device__ __forceinline__ void max_into(unsigned* addr, unsigned v) {
  if (__ldcg(addr) < v) atomicMax(addr, v);
}

// |x_i|^2 (fp64 accumulate -> fp32) and the global maximum: the SIMT Gram path (tiny graphs) needs nothing else.
__global__ void __launch_bounds__(256)
sqnorm_kernel(const float* __restrict__ X, int n, int d, float* __restrict__ sq, unsigned* __restrict__ sqmax_bits) {
  const int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (row >= n) return;
  const float* x = X + (size_t)row * d;
  double s = 0.0;
  for (int c = lane; c < d; c += 32) {
    const float x0 = __ldg(x + c);
    s += (double)x0 * (double)x0;
  }
  s = warp_sum(s);
  if (lane == 0) {
    const float f = (float)s;
    sq[row] = f;
    if (f == f) max_into(sqmax_bits, __float_as_uint(f));  // non-negative floats order like their bits
  }
}

constexpr int F16_TARGET_LOG2 = 8;  // rows are scaled to a norm in [0.58, 1.16) * 2^8

// fp16 operands of the tensor-core Gram kernel (knn_tc.cu), fused with the norms so that X is read from HBM once: row i is
// scaled by 2^-E_i to a norm in [148, 296) (exact; no fp16 overflow, and fp16's subnormal range lies 2^-22 below the row's
// own norm), then hi = fp16(z) and -- two-pass mode only, L != NULL -- lo = fp16(z - hi); row stride d_pad, zero padded.
// rscale[i] = 2^E_i undoes the scaling in the Gram epilogue.  Also the largest operand residual
// rho = max_j |x_j - hi_j 2^E_j|_2 (exact in fp64, rounded up), which bounds the Gram error: one pass computes hi_i . hi_j
// (error <= rho (|x_i| + |x_j| + rho)), two passes (hi + lo)_i . hi_j (error <= |x_i| rho + O(2^-22)); small[5] tells
// knn_err_bound() which.  NREG > 0: the row (d_pad <= 64 NREG) is held in registers, one sweep over X; NREG = 0: any d, the
// second sweep hits L1.
template <int NREG>
__global__ void __launch_bounds__(256)
sqnorm_split_f16_kernel(const float* __restrict__ X, int n, int d, int d_pad, float* __restrict__ sq, unsigned* __restrict__ small,
                        __half* __restrict__ H, __half* __restrict__ L, float* __restrict__ rscale, unsigned* __restrict__ thr_g) {
  // the four global maxima (|x|^2, rho, range of E) are reduced per CTA first: 10 k warps reading and bumping the same
  // 32-byte sector of L2 one after the other cost more than the rest of the kernel
  __shared__ unsigned sh_max[4][8];
  // A warp takes TWO rows (NREG > 0) and has both rows' loads in flight before it touches either: the kernel is one HBM round
  // trip plus two butterflies per row, and with a row per warp the C2 grid was 1.1 waves of CTAs (25 us cold for 32 MB).
  constexpr int RPW = (NREG > 0) ? 2 : 1;
  const int warp_g = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  const bool vec2 = (d & 1) == 0;  // float2 loads need an 8-byte aligned row
  float2 xr[RPW][NREG > 0 ? NREG : 1];
  int rows_i[RPW];
  bool lives[RPW];
#pragma unroll
  for (int q = 0; q < RPW; ++q) {
    const int row_raw = warp_g * RPW + q;
    lives[q] = row_raw < n;
    rows_i[q] = lives[q] ? row_raw : n - 1;  // idle slots of the last CTA recompute the last row and store nothing
    if (NREG > 0) {
      const float* x = X + (size_t)rows_i[q] * d;
#pragma unroll
      for (int t = 0; t < NREG; ++t) {
        const int c = 2 * lane + 64 * t;
        float2 v = make_float2(0.f, 0.f);
        if (vec2) {
          if (c < d) v = __ldg(reinterpret_cast<const float2*>(x + c));
        } else {
          if (c < d) v.x = __ldg(x + c);
          if (c + 1 < d) v.y = __ldg(x + c + 1);
        }
        xr[q][t] = v;
      }
    }
  }
  unsigned mx_f = 0u, mx_rho = 0u, mx_e = 0u, mx_ne = 0u;
#pragma unroll
  for (int q = 0; q < RPW; ++q) {
    const int row = rows_i[q];
    const bool live = lives[q];
    const float* x = X + (size_t)row * d;
    double s = 0.0;
    if (NREG > 0) {
#pragma unroll
      for (int t = 0; t < NREG; ++t) {
        s += (double)xr[q][t].x * (double)xr[q][t].x;
        s += (double)xr[q][t].y * (double)xr[q][t].y;
      }
    } else {
      for (int c = 2 * lane; c < d; c += 64) {
        const float x0 = __ldg(x + c);
        const float x1 = (c + 1 < d) ? __ldg(x + c + 1) : 0.f;
        s += (double)x0 * (double)x0;
        s += (double)x1 * (double)x1;
      }
    }
    s = warp_sum(s);
    // E_i from the row NORM, with the bucket boundaries at |x|^2 = 2^k / 1.5 so that rows normalised to 1 (every caller of the
    // layer) all get the same E whatever their rounding: 2^(2F - 1) <= 1.5 |x_i|^2 < 2^(2F + 1), E = F - 8, hence
    // 148 <= |z_i| < 296.  The target norm 2^8 (not 1) keeps `lo` = z - hi a NORMAL fp16 number for every element above
    // 2^-11 |x_i| and hi's own subnormal range 2^-22 below the row norm; |z_ik| < 296 is far from fp16's 65504.
    int E = -F16_TARGET_LOG2;
    {
      const unsigned b = __float_as_uint((float)(1.5 * s));
      const int ex = (int)((b >> 23) & 0xFFu);
      if (b != 0u && ex != 0xFF) E = min(60, max(-60, ((ex - 127 + 1) >> 1) - F16_TARGET_LOG2));  // arithmetic shift = floor
    }
    double r2 = 0.0;
    const float down = ldexpf(1.f, -E);  // |E| <= 60: both factors are normal numbers, the products below are exact
    const double up = ldexp(1.0, E);
    auto emit = [&](int c, float x0, float x1) {
      const float z0 = x0 * down, z1 = x1 * down;
      const __half h0 = __float2half_rn(z0), h1 = __float2half_rn(z1);
      const float f0 = __half2float(h0), f1 = __half2float(h1);
      __half2 hv;
      hv.x = h0;
      hv.y = h1;
      if (live) *reinterpret_cast<__half2*>(H + (size_t)row * d_pad + c) = hv;
      if (live && L != nullptr) {
        __half2 lv;
        lv.x = __float2half_rn(z0 - f0);
        lv.y = __float2half_rn(z1 - f1);
        *reinterpret_cast<__half2*>(L + (size_t)row * d_pad + c) = lv;
      }
      const double e0 = (double)x0 - (double)f0 * up, e1 = (double)x1 - (double)f1 * up;
      r2 += e0 * e0 + e1 * e1;
    };
    if (NREG > 0) {
#pragma unroll
      for (int t = 0; t < NREG; ++t) {
        const int c = 2 * lane + 64 * t;
        if (c < d_pad) emit(c, xr[q][t].x, xr[q][t].y);
      }
    } else {
      for (int c = 2 * lane; c < d_pad; c += 64) {  // second sweep over the row: L1 hits
        const float x0 = (c < d) ? __ldg(x + c) : 0.f;
        const float x1 = (c + 1 < d) ? __ldg(x + c + 1) : 0.f;
        emit(c, x0, x1);
      }
    }
    r2 = warp_sum(r2);
    const float f = (float)s;
    const float rho = __double2float_ru(sqrt(r2) * 1.000001);
    if (lane == 0 && live) {
      sq[row] = f;
      rscale[row] = ldexpf(1.f, E);
      if (thr_g != nullptr) thr_g[row] = 0xFF800000u;  // float_to_ordered(+inf): the row's shared threshold (knn_tc.cu)
      if (row == 0) small[5] = (L != nullptr) ? 1u : 2u;  // operand sides whose rounding rho has to cover (knn_err_bound)
    }
    mx_f = max(mx_f, (f == f) ? __float_as_uint(f) : 0u);      // non-negative floats order like their bits
    mx_rho = max(mx_rho, (rho == rho) ? __float_as_uint(rho) : 0u);
    mx_e = max(mx_e, (unsigned)(E + 128));         // range of the row scales: when all rows share one scale (normalised
    mx_ne = max(mx_ne, 255u - (unsigned)(E + 128));  // features) the Gram epilogue skips the per-row / per-column factors
  }
  const int warp = threadIdx.x >> 5;
  if (lane == 0) {
    sh_max[0][warp] = mx_f;
    sh_max[1][warp] = mx_rho;
    sh_max[2][warp] = mx_e;
    sh_max[3][warp] = mx_ne;
  }
  __syncthreads();
  if (warp == 0) {
    const unsigned v = sh_max[lane >> 3][lane & 7];  // lane = 8 * quantity + warp
    unsigned m = v;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(FULL, m, o));
    if ((lane & 7) == 0) max_into(small + (lane == 0 ? 0 : 1 + (lane >> 3)), m);  // small[0], [2], [3], [4]
  }
}

template <bool VEC4>
__device__ __forceinline__ void load_tile_regs(const float* __restrict__ X, int n, int d, int rbase, int k0, int tid,
                                               float4 (&reg)[2]) {
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    int f = tid + t * GEMM_THREADS;
    int r = f >> 2, kq = f & 3;
    int gi = rbase + r, gk = k0 + kq * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (gi < n) {
      const float* p = X + (size_t)gi * d + gk;
      if (VEC4) {
        if (gk < d) v = __ldg(reinterpret_cast<const float4*>(p));
      } else {
        if (gk + 0 < d) v.x = __ldg(p + 0);
        if (gk + 1 < d) v.y = __ldg(p + 1);
        if (gk + 2 < d) v.z = __ldg(p + 2);
        if (gk + 3 < d) v.w = __ldg(p + 3);
      }
    }
    reg[t] = v;
  }
}

__device__ __forceinline__ void store_tile_smem(float* __restrict__ S, int lds, int tid, const float4 (&reg)[2]) {
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    int f = tid + t * GEMM_THREADS;
    int r = f >> 2, kq = f & 3;
    S[(kq * 4 + 0) * lds + r] = reg[t].x;
    S[(kq * 4 + 1) * lds + r] = reg[t].y;
    S[(kq * 4 + 2) * lds + r] = reg[t].z;
    S[(kq * 4 + 3) * lds + r] = reg[t].w;
  }
}

// grid: (row tiles, column splits).  cand: [n][splits][KC] sorted keys.
// SEG: segmented search, row i only sees the columns win[i]; the splits divide the union of the row tile's windows.
template <bool VEC4, bool SEG>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
knn_gemm_topk_kernel(const float* __restrict__ X, const float* __restrict__ sq, int n, int d, int cols_per_split,
                     int splits, u64* __restrict__ cand, int row_begin, int row_end, const int2* __restrict__ win) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* As = reinterpret_cast<float*>(smem_raw);
  float* Bs = As + 2 * BK * LDS_A;
  u64* topk = reinterpret_cast<u64*>(Bs + 2 * BK * LDS_B);
  u64* pend = topk + BM * KC;
  float* thr = reinterpret_cast<float*>(pend + BM * BN);
  int* pcnt = reinterpret_cast<int*>(thr + BM);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tx = tid & 15, ty = tid >> 4;
  const int row0 = row_begin + blockIdx.x * BM;
  const int split = blockIdx.y;
  int t_lo = 0, t_hi = n;  // columns any row of the tile may see
  if (SEG) {
    t_lo = __ldg(&win[row0].x);
    t_hi = __ldg(&win[min(row_end, row0 + BM) - 1].y);
  }
  const int c_begin = t_lo + split * cols_per_split;  // a split past the windows runs no tile and writes empty lists
  const int c_end = min(t_hi, c_begin + cols_per_split);

  for (int t = tid; t < BM * KC; t += GEMM_THREADS) topk[t] = KEY_INF;
  for (int t = tid; t < BM; t += GEMM_THREADS) {
    thr[t] = INFINITY;
    pcnt[t] = 0;
  }
  __syncthreads();

  const int ktiles = (d + BK - 1) / BK;
  for (int c0 = c_begin; c0 < c_end; c0 += BN) {
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    float4 ra[2], rb[2];
    load_tile_regs<VEC4>(X, n, d, row0, 0, tid, ra);
    load_tile_regs<VEC4>(X, n, d, c0, 0, tid, rb);
    store_tile_smem(As, LDS_A, tid, ra);
    store_tile_smem(Bs, LDS_B, tid, rb);
    __syncthreads();
    for (int kt = 0; kt < ktiles; ++kt) {
      const int cur = kt & 1;
      if (kt + 1 < ktiles) {
        load_tile_regs<VEC4>(X, n, d, row0, (kt + 1) * BK, tid, ra);
        load_tile_regs<VEC4>(X, n, d, c0, (kt + 1) * BK, tid, rb);
      }
      const float* A = As + cur * BK * LDS_A;
      const float* B = Bs + cur * BK * LDS_B;
#pragma unroll
      for (int kk = 0; kk < BK; ++kk) {
        float4 a0 = *reinterpret_cast<const float4*>(A + kk * LDS_A + ty * 4);
        float4 a1 = *reinterpret_cast<const float4*>(A + kk * LDS_A + 64 + ty * 4);
        float4 b0 = *reinterpret_cast<const float4*>(B + kk * LDS_B + tx * 4);
        float4 b1 = *reinterpret_cast<const float4*>(B + kk * LDS_B + 64 + tx * 4);
        float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      if (kt + 1 < ktiles) {
        store_tile_smem(As + (cur ^ 1) * BK * LDS_A, LDS_A, tid, ra);
        store_tile_smem(Bs + (cur ^ 1) * BK * LDS_B, LDS_B, tid, rb);
      }
      __syncthreads();
    }

    // ---- fused epilogue: threshold filter, survivors appended to the row's pending list ----
    float sqj[8];
    int gjv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int cc = (j < 4) ? tx * 4 + j : 64 + tx * 4 + (j - 4);
      gjv[j] = c0 + cc;
      sqj[j] = (gjv[j] < c_end) ? __ldg(sq + gjv[j]) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int rr = (i < 4) ? ty * 4 + i : 64 + ty * 4 + (i - 4);
      int gi = row0 + rr;
      if (gi >= row_end) continue;
      float t = thr[rr];
      float sqi = __ldg(sq + gi);
      int w_lo = 0, w_hi = n;
      if (SEG) {
        const int2 w = __ldg(win + gi);
        w_lo = w.x;
        w_hi = w.y;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (gjv[j] < c_end && gjv[j] != gi && (!SEG || (gjv[j] >= w_lo && gjv[j] < w_hi))) {
          float dist = fmaf(-2.f, acc[i][j], sqi + sqj[j]);
          if (dist < t) {
            int p = atomicAdd(&pcnt[rr], 1);
            pend[rr * BN + p] = make_key(dist, gjv[j]);
          }
        }
      }
    }
    __syncthreads();
    // ---- drain: each warp folds the pending entries of its 16 rows into the sorted top-KC lists ----
    for (int rr = warp * (BM / 8); rr < (warp + 1) * (BM / 8); ++rr) {
      int c = pcnt[rr];
      if (c > 0) {
        u64 mine = topk[rr * KC + lane];
        for (int t = 0; t < c; ++t) list_insert(mine, pend[rr * BN + t], lane);
        topk[rr * KC + lane] = mine;
        if (lane == KC - 1) thr[rr] = (mine == KEY_INF) ? INFINITY : key_dist(mine);
        if (lane == 0) pcnt[rr] = 0;
      }
    }
    __syncthreads();
  }

  for (int rr = warp * (BM / 8); rr < (warp + 1) * (BM / 8); ++rr) {
    int gi = row0 + rr;
    if (gi < row_end) cand[((size_t)gi * splits + split) * KC + lane] = topk[rr * KC + lane];
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------
// rerank + completeness proof + fallback (shared with the tensor-core path)
// ---------------------------------------------------------------------------------------------------------
namespace {

constexpr int RERANK_WARPS = 4;

template <bool VEC4>
__device__ __forceinline__ double exact_d2(const float* __restrict__ xi_s, const float* __restrict__ xj, int d,
                                           int lane) {
  double part = 0.0;
  if (VEC4) {
    const float4* a = reinterpret_cast<const float4*>(xi_s);
    const float4* b = reinterpret_cast<const float4*>(xj);
    int q = d >> 2;
#pragma unroll 4
    for (int t = lane; t < q; t += 32) {
      float4 u = a[t], v = __ldg(b + t);
      double d0 = (double)u.x - (double)v.x, d1 = (double)u.y - (double)v.y;
      double d2 = (double)u.z - (double)v.z, d3 = (double)u.w - (double)v.w;
      part += d0 * d0;
      part += d1 * d1;
      part += d2 * d2;
      part += d3 * d3;
    }
  } else {
#pragma unroll 4
    for (int t = lane; t < d; t += 32) {
      double df = (double)xi_s[t] - (double)__ldg(xj + t);
      part += df * df;
    }
  }
  return warp_sum(part);  // xor butterfly: identical on all lanes, and exact_d2(i,j) == exact_d2(j,i) bitwise
}

// Row x_i held in registers as doubles (d <= 512, 16-byte aligned rows): lane owns float4 chunks lane, lane+32, lane+64,
// lane+96.  One fp32->fp64 conversion per element in the candidate loop (the conversion unit bounds this kernel) and no
// shared-memory traffic.  Same summation order as exact_d2, so the two are bitwise interchangeable.
__device__ __forceinline__ double exact_d2_reg(const double (&xr)[16], const float* __restrict__ xj, int q, int lane) {
  const float4* b = reinterpret_cast<const float4*>(xj);
  float4 v[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) v[t] = (lane + 32 * t < q) ? __ldg(b + lane + 32 * t) : make_float4(0.f, 0.f, 0.f, 0.f);
  double part = 0.0;
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    if (lane + 32 * t < q) {
      const double d0 = xr[4 * t + 0] - (double)v[t].x, d1 = xr[4 * t + 1] - (double)v[t].y;
      const double d2 = xr[4 * t + 2] - (double)v[t].z, d3 = xr[4 * t + 3] - (double)v[t].w;
      part += d0 * d0;
      part += d1 * d1;
      part += d2 * d2;
      part += d3 * d3;
    }
  }
  return warp_sum(part);
}

// |d~^2_ij - d^2_ij| <= err_coef (|x_i|^2 + max|x|^2) + 2 * [rho term].  small[0] = bits of max_j |x_j|^2, small[2] = bits of
// rho = max_j |x_j - hi_j 2^E_j|_2, the largest residual of the fp16 operands (0 on the SIMT path), small[5] = how many
// operand sides carry it: two passes, (hi + lo)_i . hi_j: |x_i| rho; one pass, hi_i . hi_j:
// |x_i . x_j - hi_i . hi_j| <= |x_i - hi_i| |x_j| + |hi_i| |x_j - hi_j| <= rho (|x_j| + |x_i| + rho).
__device__ __forceinline__ double knn_err_bound(float err_coef, float sqi, const unsigned* __restrict__ small) {
  const double sqm = (double)__uint_as_float(small[0]), rho = (double)__uint_as_float(small[2]);
  const double xi = sqrt((double)sqi);
  const double rterm = (small[5] == 2u) ? rho * (xi + sqrt(sqm) + rho) : xi * rho;
  return (double)err_coef * ((double)sqi + sqm) + 2.0 * rterm * 1.000001;
}

template <bool VEC4>
__global__ void __launch_bounds__(RERANK_WARPS * 32)
knn_rerank_kernel(const float* __restrict__ X, const float* __restrict__ sq, const unsigned* __restrict__ sqmax_bits,
                  int n, int d, int k, int row_end, CandLayout lay, const u64* __restrict__ cand, float err_coef,
                  int* __restrict__ knn_idx, float* __restrict__ knn_dist, int* __restrict__ flag_count,
                  int* __restrict__ flag_rows, int force_rows) {
  extern __shared__ __align__(16) float xs[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = lay.row_begin + blockIdx.x * RERANK_WARPS + warp;
  if (i >= row_end) return;
  float* xi = xs + (size_t)warp * d;
  const bool use_reg = VEC4 && d <= 512;
  double xr[16];
  if (use_reg) {
    const float4* xrow = reinterpret_cast<const float4*>(X + (size_t)i * d);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float4 u = (lane + 32 * t < (d >> 2)) ? __ldg(xrow + lane + 32 * t) : make_float4(0.f, 0.f, 0.f, 0.f);
      xr[4 * t + 0] = (double)u.x;
      xr[4 * t + 1] = (double)u.y;
      xr[4 * t + 2] = (double)u.z;
      xr[4 * t + 3] = (double)u.w;
    }
  } else {
    for (int t = lane; t < d; t += 32) xi[t] = X[(size_t)i * d + t];
  }

  u64 mine = KEY_INF;
  const int splits = cand_lists(lay, i);
  if (splits == 1 && lay.tc == 0) {
    mine = cand[(size_t)i * lay.stride * KC + lane];  // SIMT lists are sorted
  } else {
    for (int s = 0; s < splits; ++s) {  // tensor-core lists are unsorted sets: merge by insertion
      list_merge_set(mine, cand[((size_t)i * lay.stride + s) * KC + lane], lane);
    }
  }
  u64 last = __shfl_sync(FULL, mine, KC - 1);
  const float lower = (last == KEY_INF) ? INFINITY : key_dist(last);  // every non-candidate has d~^2 >= lower
  __syncwarp();

  // Candidates whose approximate distance exceeds the (k-1)-th approximate distance by more than twice the error bound
  // cannot be among the k-1 nearest (k-1 others are provably closer): their exact distance is not needed.
  const double errb = knn_err_bound(err_coef, sq[i], sqmax_bits);
  const u64 kth = __shfl_sync(FULL, mine, k - 2);
  const float cutoff = (kth == KEY_INF) ? INFINITY : (float)((double)key_dist(kth) + 2.0 * errb + 1e-30) * (1.f + 1e-6f);
  double myd2 = INFINITY;
  int myj = -1;
  for (int c = 0; c < KC; ++c) {
    u64 kc = __shfl_sync(FULL, mine, c);
    if (kc == KEY_INF) break;
    if (c > k - 2 && key_dist(kc) > cutoff) break;  // sorted: everything behind is farther still
    int j = key_idx(kc);
    double v = use_reg ? exact_d2_reg(xr, X + (size_t)j * d, d >> 2, lane) : exact_d2<VEC4>(xi, X + (size_t)j * d, d, lane);
    if (lane == c) {
      myd2 = v;
      myj = j;
    }
  }
  int rank = 0;
  for (int c = 0; c < KC; ++c) {
    double od = __shfl_sync(FULL, myd2, c);
    int oj = __shfl_sync(FULL, myj, c);
    if (oj >= 0 && (od < myd2 || (od == myd2 && oj < myj))) ++rank;
  }
  if (myj >= 0 && rank < k - 1) {
    knn_idx[(size_t)i * k + 1 + rank] = myj;
    knn_dist[(size_t)i * k + 1 + rank] = (float)sqrt(myd2);
  }
  if (lane == 0) {
    knn_idx[(size_t)i * k] = i;
    knn_dist[(size_t)i * k] = 0.f;
  }
  // completeness proof
  unsigned who = __ballot_sync(FULL, myj >= 0 && rank == k - 2);
  bool ok = false;
  if (who) {
    double dk = __shfl_sync(FULL, myd2, __ffs(who) - 1);
    ok = ((double)lower - errb > dk) || (lower == INFINITY);
  }
  if (i - lay.row_begin < force_rows) ok = false;  // GLL_B200_KNN_FORCE_FALLBACK (tests): treat the first rows as unproven
  if (!ok && lane == 0) {
    int p = atomicAdd(flag_count, 1);
    flag_rows[p] = i;
  }
}

constexpr int FB_WARPS = 8;

__device__ __forceinline__ void list_insert_d(double& md, int& mj, double xd, int xj, int lane) {
  bool lt = (md < xd) || (md == xd && mj < xj);
  int pos = __popc(__ballot_sync(FULL, lt));
  double pd = __shfl_up_sync(FULL, md, 1);
  int pj = __shfl_up_sync(FULL, mj, 1);
  if (lane > pos) {
    md = pd;
    mj = pj;
  } else if (lane == pos) {
    md = xd;
    mj = xj;
  }
}

// Merge the ascending 32-list (od, oj) into the ascending 32-list (md, mj), one (distance, index) pair per lane, padding
// (INFINITY, 0x7fffffff) at the end: min(A[i], B[31 - i]) holds the 32 smallest of the union as a bitonic sequence, five
// compare-exchange steps put it in order.  Replaces up to 32 serial insertions per list.
__device__ __forceinline__ bool pair_less(double ad, int aj, double bd, int bj) { return ad < bd || (ad == bd && aj < bj); }
__device__ __forceinline__ void dlist_merge_sorted(double& md, int& mj, double od, int oj, int lane) {
  const double rd = __shfl_sync(FULL, od, 31 - lane);
  const int rj = __shfl_sync(FULL, oj, 31 - lane);
  if (pair_less(rd, rj, md, mj)) {
    md = rd;
    mj = rj;
  }
#pragma unroll
  for (int j = 16; j >= 1; j >>= 1) {
    const double pd = __shfl_xor_sync(FULL, md, j);
    const int pj = __shfl_xor_sync(FULL, mj, j);
    const bool keep_min = (lane & j) == 0;
    const bool p_less = pair_less(pd, pj, md, mj);
    if (p_less == keep_min) {
      md = pd;
      mj = pj;
    }
  }
}

template <bool VEC4>
__global__ void __launch_bounds__(FB_WARPS * 32)
knn_fallback_kernel(const float* __restrict__ X, int n, int d, int k, const int* __restrict__ flag_count,
                    const int* __restrict__ flag_rows, int* __restrict__ knn_idx, float* __restrict__ knn_dist,
                    int* __restrict__ info, const int2* __restrict__ win) {
  extern __shared__ __align__(16) float xs[];
  __shared__ double sd[FB_WARPS][32];
  __shared__ int sj[FB_WARPS][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nflag = *flag_count;
  if (blockIdx.x == 0 && threadIdx.x == 0 && info != nullptr) {
    info[GLL_INFO_KNN_FALLBACK_ROWS] = nflag;
    if (nflag > 0) atomicOr(&info[GLL_INFO_STATUS], GLL_STATUS_KNN_FALLBACK);
  }
  for (int f = blockIdx.x; f < nflag; f += gridDim.x) {
    const int i = flag_rows[f];
    const int2 w = (win != nullptr) ? win[i] : make_int2(0, n);  // a segmented search scans the row's own segment
    for (int t = threadIdx.x; t < d; t += blockDim.x) xs[t] = X[(size_t)i * d + t];
    __syncthreads();
    // k - 1 <= 32 neighbours fit one 32-wide list; larger k takes a second scan that only admits pairs beyond the 32nd
    // (distance, index) of the first scan
    double ex_d = -1.0;
    int ex_j = -1;
    for (int pass = 0; pass * 32 < k - 1; ++pass) {
      double md = INFINITY;
      int mj = 0x7fffffff;
      for (int j = w.x + warp; j < w.y; j += FB_WARPS) {
        if (j == i) continue;
        double v = exact_d2<VEC4>(xs, X + (size_t)j * d, d, lane);
        if (v > ex_d || (v == ex_d && j > ex_j)) list_insert_d(md, mj, v, j, lane);
      }
      sd[warp][lane] = md;
      sj[warp][lane] = mj;
      __syncthreads();
      if (warp == 0) {
        for (int w = 1; w < FB_WARPS; ++w)
          for (int t = 0; t < 32; ++t) {
            int xj = sj[w][t];
            if (xj == 0x7fffffff) break;
            list_insert_d(md, mj, sd[w][t], xj, lane);
          }
        const int slot = pass * 32 + lane;
        if (slot < k - 1 && mj != 0x7fffffff) {
          knn_idx[(size_t)i * k + 1 + slot] = mj;
          knn_dist[(size_t)i * k + 1 + slot] = (float)sqrt(md);
        }
        if (lane == 0 && pass == 0) {
          knn_idx[(size_t)i * k] = i;
          knn_dist[(size_t)i * k] = 0.f;
        }
        if (lane == 31) {  // threshold for the next scan
          sd[0][0] = md;
          sj[0][0] = mj;
        }
      }
      __syncthreads();
      ex_d = sd[0][0];
      ex_j = sj[0][0];
      __syncthreads();
    }
    __syncthreads();
  }
}

// ---- brute-force fallback for k - 1 <= 32, fast for FEW rows: the flagged rows' column ranges are dealt to all CTAs ----
// (a flagged row used to be one CTA's job: 171 ms for two rows of a 1M-node graph.)  Task t = (flagged row f, column chunk c)
// with C = max(1, G / nflag) chunks per row; every task leaves the 32 smallest (exact fp64 distance, index) pairs of its
// chunk; with C == 1 that is the row's answer, otherwise the last CTA to finish merges the C lists of every row.
template <bool VEC4>
__global__ void __launch_bounds__(FB_WARPS * 32)
knn_fallback_scan_kernel(const float* __restrict__ X, int n, int d, int k, const int* __restrict__ flag_count,
                         const int* __restrict__ flag_rows, int* __restrict__ knn_idx, float* __restrict__ knn_dist,
                         int* __restrict__ info, double* __restrict__ part_d, int* __restrict__ part_j,
                         unsigned* __restrict__ ticket, const int2* __restrict__ win) {
  extern __shared__ __align__(16) float xs[];
  __shared__ double sd[FB_WARPS][32];
  __shared__ int sj[FB_WARPS][32];
  __shared__ int last_cta;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nflag = *flag_count;
  if (blockIdx.x == 0 && threadIdx.x == 0 && info != nullptr) {
    info[GLL_INFO_KNN_FALLBACK_ROWS] = nflag;
    if (nflag > 0) atomicOr(&info[GLL_INFO_STATUS], GLL_STATUS_KNN_FALLBACK);
  }
  if (nflag == 0) return;
  const int G = gridDim.x, C = max(1, min(128, G / nflag));  // <= 128 chunks per row: the serial merge stays short
  const long long T = (long long)nflag * C;
  for (long long t = blockIdx.x; t < T; t += G) {
    const int f = (int)(t / C), c = (int)(t - (long long)f * C);
    const int i = flag_rows[f];
    const int2 w = (win != nullptr) ? win[i] : make_int2(0, n);  // a segmented search scans the row's own segment
    const int j0 = w.x + (int)((long long)(w.y - w.x) * c / C), j1 = w.x + (int)((long long)(w.y - w.x) * (c + 1) / C);
    __syncthreads();  // the previous task's readers of xs / sd / sj are done
    for (int q = threadIdx.x; q < d; q += blockDim.x) xs[q] = X[(size_t)i * d + q];
    __syncthreads();
    double md = INFINITY, thr_d = INFINITY;
    int mj = 0x7fffffff, thr_j = 0x7fffffff;
    // four columns per trip: their row loads and butterflies are independent (one column at a time is a chain of L2 round trips)
    for (int jb = j0 + 4 * warp; jb < j1; jb += 4 * FB_WARPS) {
      double v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = min(jb + u, j1 - 1);  // clamped duplicates are dropped below
        v[u] = exact_d2<VEC4>(xs, X + (size_t)j * d, d, lane);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = jb + u;
        if (j >= j1 || j == i) continue;
        if (v[u] < thr_d || (v[u] == thr_d && j < thr_j)) {  // warp-uniform: only pairs that enter the list pay for the insertion
          list_insert_d(md, mj, v[u], j, lane);
          thr_d = __shfl_sync(FULL, md, 31);
          thr_j = __shfl_sync(FULL, mj, 31);
        }
      }
    }
    sd[warp][lane] = md;
    sj[warp][lane] = mj;
    __syncthreads();
    if (warp == 0) {
      for (int w = 1; w < FB_WARPS; ++w) dlist_merge_sorted(md, mj, sd[w][lane], sj[w][lane], lane);
      if (C == 1) {
        if (lane < k - 1 && mj != 0x7fffffff) {
          knn_idx[(size_t)i * k + 1 + lane] = mj;
          knn_dist[(size_t)i * k + 1 + lane] = (float)sqrt(md);
        }
        if (lane == 0) {
          knn_idx[(size_t)i * k] = i;
          knn_dist[(size_t)i * k] = 0.f;
        }
      } else {
        part_d[(size_t)t * 32 + lane] = md;
        part_j[(size_t)t * 32 + lane] = mj;
      }
    }
  }
  if (C == 1) return;
  // the last CTA to finish merges the C chunk lists of every flagged row: its eight warps take C / 8 lists each (the loads of
  // a warp's lists are issued together), then warp 0 merges the eight partial lists
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    last_cta = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (!last_cta) return;
  __threadfence();
  if (C <= 16) {  // many flagged rows, few chunks each: one warp per row
    for (int f = warp; f < nflag; f += FB_WARPS) {
      const int i = flag_rows[f];
      double md = INFINITY;
      int mj = 0x7fffffff;
      for (int c0 = 0; c0 < C; c0 += 4) {
        double ld[4];
        int lj[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int c = c0 + u;
          ld[u] = (c < C) ? __ldcg(part_d + ((size_t)f * C + c) * 32 + lane) : INFINITY;
          lj[u] = (c < C) ? __ldcg(part_j + ((size_t)f * C + c) * 32 + lane) : 0x7fffffff;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) dlist_merge_sorted(md, mj, ld[u], lj[u], lane);
      }
      if (lane < k - 1 && mj != 0x7fffffff) {
        knn_idx[(size_t)i * k + 1 + lane] = mj;
        knn_dist[(size_t)i * k + 1 + lane] = (float)sqrt(md);
      }
      if (lane == 0) {
        knn_idx[(size_t)i * k] = i;
        knn_dist[(size_t)i * k] = 0.f;
      }
    }
    return;
  }
  for (int f = 0; f < nflag; ++f) {
    const int i = flag_rows[f];
    double md = INFINITY;
    int mj = 0x7fffffff;
    for (int c0 = warp; c0 < C; c0 += 4 * FB_WARPS) {
      double ld[4];
      int lj[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int c = c0 + u * FB_WARPS;
        ld[u] = (c < C) ? __ldcg(part_d + ((size_t)f * C + c) * 32 + lane) : INFINITY;
        lj[u] = (c < C) ? __ldcg(part_j + ((size_t)f * C + c) * 32 + lane) : 0x7fffffff;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) dlist_merge_sorted(md, mj, ld[u], lj[u], lane);
    }
    __syncthreads();
    sd[warp][lane] = md;
    sj[warp][lane] = mj;
    __syncthreads();
    if (warp == 0) {
      for (int w = 1; w < FB_WARPS; ++w) dlist_merge_sorted(md, mj, sd[w][lane], sj[w][lane], lane);
      if (lane < k - 1 && mj != 0x7fffffff) {
        knn_idx[(size_t)i * k + 1 + lane] = mj;
        knn_dist[(size_t)i * k + 1 + lane] = (float)sqrt(md);
      }
      if (lane == 0) {
        knn_idx[(size_t)i * k] = i;
        knn_dist[(size_t)i * k] = 0.f;
      }
    }
  }
}


// ---------------------------------------------------------------------------------------------------------
// k in (33, 64]: two candidate rounds of 32 (the second excludes the first by key), merged and re-ranked together.
// Used by the evaluation path (utils.laplace asks for k = 50, utils.py:651); the layer itself uses k = 25.
// ---------------------------------------------------------------------------------------------------------
// one warp per row: union of the row's candidate sets of one round -> one sorted 32-list; optionally its last key
__global__ void __launch_bounds__(RERANK_WARPS * 32)
knn_merge_kernel(int row_end, CandLayout lay, const u64* __restrict__ cand, u64* __restrict__ merged, u64* __restrict__ excl) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = lay.row_begin + blockIdx.x * RERANK_WARPS + warp;
  if (i >= row_end) return;
  const int splits = cand_lists(lay, i);
  u64 mine = KEY_INF;
  for (int s = 0; s < splits; ++s) {
    list_merge_set(mine, cand[((size_t)i * lay.stride + s) * KC + lane], lane);
  }
  merged[(size_t)(i - lay.row_begin) * KC + lane] = mine;
  if (excl != nullptr && lane == KC - 1) excl[i] = mine;  // KEY_INF if fewer than 32 columns exist: round 2 finds nothing
}

template <bool VEC4>
__global__ void __launch_bounds__(RERANK_WARPS * 32)
knn_rerank64_kernel(const float* __restrict__ X, const float* __restrict__ sq, const unsigned* __restrict__ sqmax_bits, int n, int d,
                    int k, int row_begin, int row_end, const u64* __restrict__ m1, const u64* __restrict__ m2, float err_coef,
                    int* __restrict__ knn_idx, float* __restrict__ knn_dist, int* __restrict__ flag_count,
                    int* __restrict__ flag_rows, int force_rows) {
  extern __shared__ __align__(16) float xs[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = row_begin + blockIdx.x * RERANK_WARPS + warp;
  if (i >= row_end) return;
  float* xi = xs + (size_t)warp * d;
  for (int t = lane; t < d; t += 32) xi[t] = X[(size_t)i * d + t];
  __syncwarp();
  const u64 ca = m1[(size_t)(i - row_begin) * KC + lane];
  u64 cb = m2[(size_t)(i - row_begin) * KC + lane];
  const u64 last = __shfl_sync(FULL, cb, KC - 1);
  const float lower = (last == KEY_INF) ? INFINITY : key_dist(last);  // every non-candidate has d~^2 >= lower
  // the second round re-admits first-round members whose stored value ties with the first round's 32nd (knn_tc.cu): drop them
  {
    bool dup = false;
    for (int c = 0; c < KC; ++c) {
      const u64 oa = __shfl_sync(FULL, ca, c);
      dup |= (oa != KEY_INF && cb != KEY_INF && key_idx(oa) == key_idx(cb));
    }
    if (dup) cb = KEY_INF;
  }
  double da = INFINITY, db = INFINITY;
  int ja = -1, jb = -1;
  for (int c = 0; c < 2 * KC; ++c) {
    const u64 kc = __shfl_sync(FULL, (c < KC) ? ca : cb, c & (KC - 1));
    if (kc == KEY_INF) continue;
    const int j = key_idx(kc);
    const double v = exact_d2<VEC4>(xi, X + (size_t)j * d, d, lane);
    if (lane == (c & (KC - 1))) {
      if (c < KC) {
        da = v;
        ja = j;
      } else {
        db = v;
        jb = j;
      }
    }
  }
  int ra = 0, rb = 0;
  for (int c = 0; c < 2 * KC; ++c) {
    const double od = __shfl_sync(FULL, (c < KC) ? da : db, c & (KC - 1));
    const int oj = __shfl_sync(FULL, (c < KC) ? ja : jb, c & (KC - 1));
    if (oj < 0) continue;
    ra += (od < da || (od == da && oj < ja)) ? 1 : 0;
    rb += (od < db || (od == db && oj < jb)) ? 1 : 0;
  }
  if (ja >= 0 && ra < k - 1) {
    knn_idx[(size_t)i * k + 1 + ra] = ja;
    knn_dist[(size_t)i * k + 1 + ra] = (float)sqrt(da);
  }
  if (jb >= 0 && rb < k - 1) {
    knn_idx[(size_t)i * k + 1 + rb] = jb;
    knn_dist[(size_t)i * k + 1 + rb] = (float)sqrt(db);
  }
  if (lane == 0) {
    knn_idx[(size_t)i * k] = i;
    knn_dist[(size_t)i * k] = 0.f;
  }
  // completeness proof against the (k-1)-th exact distance
  const unsigned wa = __ballot_sync(FULL, ja >= 0 && ra == k - 2), wb = __ballot_sync(FULL, jb >= 0 && rb == k - 2);
  bool ok = false;
  if (wa | wb) {
    const double dk = wa ? __shfl_sync(FULL, da, __ffs(wa) - 1) : __shfl_sync(FULL, db, __ffs(wb) - 1);
    const double errb = knn_err_bound(err_coef, sq[i], sqmax_bits);
    ok = ((double)lower - errb > dk) || (lower == INFINITY);
  }
  if (i - row_begin < force_rows) ok = false;  // GLL_B200_KNN_FORCE_FALLBACK (tests): treat the first rows as unproven
  if (!ok && lane == 0) {
    int p = atomicAdd(flag_count, 1);
    flag_rows[p] = i;
  }
}

}  // namespace

int knn_fallback_grid() { return 2 * device_info().sms; }
size_t knn_fallback_scratch_bytes() { return align_up((size_t)knn_fallback_grid() * 32 * (sizeof(double) + sizeof(int)), 256); }

namespace {

int simt_splits(int n, int rows, int* cols_per_split) {
  // at least one row tile: size queries of shapes the search refuses (an empty row range) must not divide by zero
  int row_tiles = max(1, ceil_div(rows, BM)), col_tiles = ceil_div(n, BN);
  int want = ceil_div(2 * device_info().sms, row_tiles);
  want = max(1, min(want, min(col_tiles, KNN_MAX_SPLITS)));
  int tiles_per = ceil_div(col_tiles, want);
  *cols_per_split = tiles_per * BN;
  return ceil_div(col_tiles, tiles_per);
}

// the widest union of segment windows over a 128-row tile: the columns a SIMT row tile of a segmented search may see
int widest_tile_window(int n, const int* seg_ptr) {
  int wmax = 1;
  for (int r0 = 0, s = 0; r0 < n; r0 += BM) {
    while (seg_ptr[s + 1] <= r0) ++s;
    int t = s;
    const int r1 = min(n, r0 + BM) - 1;
    while (seg_ptr[t + 1] <= r1) ++t;
    wmax = max(wmax, seg_ptr[t + 1] - seg_ptr[s]);
  }
  return wmax;
}

// |fl(d~^2) - d^2| <= (gamma_d + 4u)(|x_i|^2 + |x_j|^2), gamma_d = d u/(1 - d u), u = 2^-24 (sequential fp32 FMA chain)
float simt_err_coef(int d) {
  const double u = 5.9604644775390625e-8;
  return (float)(((double)d * u / (1.0 - (double)d * u) + 4.0 * u) * 1.0001);
}

// How a search over rows [row_begin, row_end) runs: the Gram path, the candidate lists it leaves and the error bound of their
// approximate distances.
struct KnnPlan {
  int row_begin, row_end;
  TcPlan tc;              // tc.ok: the tensor-core Gram path; otherwise the SIMT kernel with lay.stride column splits of cps columns
  int cps;
  CandLayout lay;         // lay.stride lists per row; lay.gfirst is set once the unit table is on the device
  float err_coef;
  std::vector<int> ints;  // segmented search: seg_ptr, then the tensor-core unit table (gfirst, gct, bstart; see SegDev)
};

// nseg > 1: the segmented search over all n rows (row_begin = 0, row_end = n); col_begin: columns before it are not searched
KnnPlan knn_plan(int n, int d, int row_begin, int row_end, int col_begin = 0, const int* seg_ptr = nullptr, int nseg = 1) {
  const bool seg = nseg > 1;
  KnnPlan p;
  p.row_begin = row_begin;
  p.row_end = row_end;
  std::vector<int> tab;
  p.tc = seg ? knn_tc_plan_segments(n, d, seg_ptr, nseg, &tab) : knn_tc_plan(n, d, row_begin, row_end, col_begin);
  memset(&p.lay, 0, sizeof(p.lay));
  p.lay.row_begin = row_begin;
  if (p.tc.ok) {
    p.cps = 0;
    p.lay.stride = p.tc.max_splits;
    p.lay.tc = p.tc.aligned ? 2 : (seg ? 3 : 1);
    p.lay.row_tile = 128 * p.tc.rstep;  // rows per row group
    p.lay.col_tiles = p.tc.col_tiles;
    p.lay.grid = p.tc.grid;
    p.lay.units = p.tc.units;
    p.err_coef = knn_tc_err_coef(d, p.tc.passes);
  } else {
    tab.clear();
    p.lay.stride = simt_splits(seg ? widest_tile_window(n, seg_ptr) : n, row_end - row_begin, &p.cps);
    p.err_coef = simt_err_coef(d);
  }
  if (seg) {
    p.ints.assign(seg_ptr, seg_ptr + nseg + 1);
    p.ints.insert(p.ints.end(), tab.begin(), tab.end());
  }
  return p;
}

// What a kNN entry takes from its workspace; the members it does not use stay NULL.
struct KnnBufs {
  float* sq;
  unsigned* small;     // small[0]: bits of max |x|^2, small[1]: flag_count, small[8]: fallback ticket (zeroed per search)
  int* flag_count;
  u64* cand;           // the plan's rows x lay.stride lists, indexed by GLOBAL row: where row 0 would live
  int* flag_rows;
  char* tc_ws;         // fp16 hi / lo operands of the tensor-core path
  unsigned* thr_g;     // per-row shared thresholds
  float* rscale;       // per-row power-of-two scale of the fp16 operands
  void* fb_scratch;    // chunk lists of the brute-force fallback
  u64* merged;         // k > 33: the two rounds' merged lists [2][rows][KC]; cached search: [n][KC]
  u64* excl;           // k > 33: the first round's 32nd key per row
  int2* win;           // segmented search: the rows' column windows
  int* ints;           // segmented search: KnnPlan::ints
  u64* cand_base;      // cached search: the base x batch-columns lists of base rows [0, p.row_begin)
};

// Sizes and carves the workspace of every kNN entry; returns the bytes needed (ws == NULL: size query only).  pb != NULL: the
// cached search, whose two candidate launches follow the tensor-core plans p and *pb (max_splits = 0 when one declines).
size_t knn_bufs(void* ws, int n, int d, int k, const KnnPlan& p, const KnnPlan* pb, KnnBufs* out) {
  Carver cv(ws, ~(size_t)0);
  const size_t rows = (size_t)(p.row_end - p.row_begin);
  const size_t stride = (size_t)(pb ? p.tc.max_splits : p.lay.stride);
  KnnBufs b;
  memset(&b, 0, sizeof(b));
  b.sq = cv.take<float>(n);
  b.small = cv.take<unsigned>(64);
  b.flag_count = reinterpret_cast<int*>(b.small + 1);
  b.cand = cv.take<u64>(rows * stride * KC) - (size_t)p.row_begin * stride * KC;
  b.flag_rows = cv.take<int>(pb ? (size_t)n : rows);
  b.tc_ws = cv.take<char>(knn_tc_ws_upper(n, d));
  b.thr_g = cv.take<unsigned>(n);
  b.rscale = cv.take<float>(n);
  b.fb_scratch = cv.take<char>(knn_fallback_scratch_bytes());
  if (k > KC + 1) {
    b.merged = cv.take<u64>(2 * rows * KC);
    b.excl = cv.take<u64>(n);
  }
  if (!p.ints.empty()) {
    b.win = cv.take<int2>(n);
    b.ints = cv.take<int>(p.ints.size());
  }
  if (pb) {
    b.cand_base = cv.take<u64>((size_t)p.row_begin * pb->tc.max_splits * KC);
    b.merged = cv.take<u64>((size_t)n * KC);
  }
  if (out) *out = b;
  return cv.off;
}

// fp32 SIMT Gram with the fused top-k epilogue; win != NULL: segmented search (column windows per row)
int launch_simt(const float* X, const float* sq, int n, int d, int cps, int splits, u64* cand, int row_begin, int row_end,
                const int2* win, cudaStream_t st) {
  const bool vec4 = (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
  const bool seg = win != nullptr;
  auto kern = vec4 ? (seg ? knn_gemm_topk_kernel<true, true> : knn_gemm_topk_kernel<true, false>)
                   : (seg ? knn_gemm_topk_kernel<false, true> : knn_gemm_topk_kernel<false, false>);
  const dim3 grid(ceil_div(row_end - row_begin, BM), splits);
  const size_t smem = gemm_smem_bytes();
  GLL_CUDA_CHECK(set_max_dynamic_smem_once((const void*)kern, (int)smem));
  {
    GLL_PROF(KID_GRAM_TOPK, st);
    kern<<<grid, GEMM_THREADS, smem, st>>>(X, sq, n, d, cps, splits, cand, row_begin, row_end, win);
  }
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

// fp16 operand split + norms: rows of up to 1024 padded columns stay in registers (one sweep over X)
int launch_split_f16(const float* X, int n, int d, const TcPlan& plan, float* sq, unsigned* small, char* tc_ws, float* rscale,
                     unsigned* thr_g, cudaStream_t st) {
  __half* H = reinterpret_cast<__half*>(tc_ws);
  __half* L = (plan.passes == 2) ? reinterpret_cast<__half*>(tc_ws + align_up((size_t)n * plan.d_pad * 2, 256)) : nullptr;
  const int grid = ceil_div((long long)ceil_div(n, plan.d_pad <= 1024 ? 2 : 1) * 32, 256);  // two rows per warp when the row fits registers
  if (plan.d_pad <= 256)
    sqnorm_split_f16_kernel<4><<<grid, 256, 0, st>>>(X, n, d, plan.d_pad, sq, small, H, L, rscale, thr_g);
  else if (plan.d_pad <= 512)
    sqnorm_split_f16_kernel<8><<<grid, 256, 0, st>>>(X, n, d, plan.d_pad, sq, small, H, L, rscale, thr_g);
  else if (plan.d_pad <= 1024)
    sqnorm_split_f16_kernel<16><<<grid, 256, 0, st>>>(X, n, d, plan.d_pad, sq, small, H, L, rscale, thr_g);
  else
    sqnorm_split_f16_kernel<0><<<grid, 256, 0, st>>>(X, n, d, plan.d_pad, sq, small, H, L, rscale, thr_g);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

// |x_i|^2 and the global max for the search, plus the fp16 operand split when the tensor-core plan runs
int launch_norms(const float* X, int n, int d, const TcPlan& plan, const KnnBufs& b, cudaStream_t st) {
  GLL_PROF(KID_SQNORM, st);
  if (plan.ok) return launch_split_f16(X, n, d, plan, b.sq, b.small, b.tc_ws, b.rscale, b.thr_g, st);
  sqnorm_kernel<<<ceil_div((long long)n * 32, 256), 256, 0, st>>>(X, n, d, b.sq, b.small);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

// Exact re-rank of rows [lay.row_begin, row_end), their completeness proof, and the brute-force search of the rows it could not
// prove.  k <= 33: the candidate lists `cand` under `lay`; k > 33: b.merged, the two rounds' merged lists.
int knn_finish(const float* X, int n, int d, int k, int row_end, const CandLayout& lay, const u64* cand, float err_coef,
               const KnnBufs& b, int* knn_idx, float* knn_dist, int* info, cudaStream_t st) {
  const bool vec4 = (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
  const bool two_rounds = k > KC + 1;
  const int row_begin = lay.row_begin, blocks = ceil_div(row_end - row_begin, RERANK_WARPS);
  const size_t smem = sizeof(float) * (size_t)RERANK_WARPS * d, fsmem = sizeof(float) * (size_t)d;
  const char* force = getenv("GLL_B200_KNN_FORCE_FALLBACK");
  const int force_rows = force ? atoi(force) : 0;
  const bool no_fallback = getenv("GLL_B200_KNN_DEBUG") != nullptr;  // timing experiments: every row would be "unproven"
  if (two_rounds) {
    auto kern = vec4 ? knn_rerank64_kernel<true> : knn_rerank64_kernel<false>;
    GLL_CUDA_CHECK(set_max_dynamic_smem_once((const void*)kern, (int)smem));
    GLL_PROF(KID_RERANK, st);
    kern<<<blocks, RERANK_WARPS * 32, smem, st>>>(X, b.sq, b.small, n, d, k, row_begin, row_end, b.merged,
                                                 b.merged + (size_t)(row_end - row_begin) * KC, err_coef, knn_idx, knn_dist,
                                                 b.flag_count, b.flag_rows, force_rows);
  } else {
    auto kern = vec4 ? knn_rerank_kernel<true> : knn_rerank_kernel<false>;
    GLL_CUDA_CHECK(set_max_dynamic_smem_once((const void*)kern, (int)smem));
    GLL_PROF(KID_RERANK, st);
    kern<<<blocks, RERANK_WARPS * 32, smem, st>>>(X, b.sq, b.small, n, d, k, row_end, lay, cand, err_coef, knn_idx, knn_dist,
                                                 b.flag_count, b.flag_rows, force_rows);
  }
  GLL_LAUNCH_CHECK();
  if (no_fallback) return GLL_OK;
  if (two_rounds) {
    auto kern = vec4 ? knn_fallback_kernel<true> : knn_fallback_kernel<false>;
    GLL_CUDA_CHECK(set_max_dynamic_smem_once((const void*)kern, (int)fsmem));
    GLL_PROF(KID_KNN_FALLBACK, st);
    kern<<<device_info().sms, FB_WARPS * 32, fsmem, st>>>(X, n, d, k, b.flag_count, b.flag_rows, knn_idx, knn_dist, info, b.win);
  } else {
    // the rows' column ranges dealt to all CTAs
    const int fblocks = knn_fallback_grid();
    double* part_d = reinterpret_cast<double*>(b.fb_scratch);
    int* part_j = reinterpret_cast<int*>(part_d + (size_t)fblocks * 32);
    auto kern = vec4 ? knn_fallback_scan_kernel<true> : knn_fallback_scan_kernel<false>;
    GLL_CUDA_CHECK(set_max_dynamic_smem_once((const void*)kern, (int)fsmem));
    GLL_PROF(KID_KNN_FALLBACK, st);
    kern<<<fblocks, FB_WARPS * 32, fsmem, st>>>(X, n, d, k, b.flag_count, b.flag_rows, knn_idx, knn_dist, info, part_d, part_j,
                                                b.small + 8, b.win);
  }
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------------------------------
// Segmented search (gll_knn_segments): independent graphs stacked as row segments; row i of segment s gets its k nearest
// neighbours among the rows of s only.  Every kernel sees the rows' column windows win[i] = [lo, hi): the Gram kernels only
// visit the column tiles that meet a row tile's windows and mask the rest per row, the fallback scans the window, and the
// re-rank is unchanged (columns outside the window never enter a set, so its completeness proof covers the window).
// ------------------------------------------------------------------------------------------------------------------------
namespace {

constexpr int UPLOAD_INTS = 1000;
struct IntChunk {
  int v[UPLOAD_INTS];
};
// host ints -> device through the kernel parameters: no host memory is read when the work runs, so the call can be captured
// in a CUDA graph (a copy from pageable host memory cannot)
__global__ void upload_ints_kernel(IntChunk c, int count, int* __restrict__ dst) {
  for (int t = threadIdx.x; t < count; t += blockDim.x) dst[t] = c.v[t];
}

// win[i] = [seg_ptr[s], seg_ptr[s + 1]) for the rows i of segment s = blockIdx.x
__global__ void seg_windows_kernel(const int* __restrict__ seg_ptr, int2* __restrict__ win) {
  const int lo = seg_ptr[blockIdx.x], hi = seg_ptr[blockIdx.x + 1];
  for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) win[i] = make_int2(lo, hi);
}

// The plain search of rows [row_begin, row_end) and (nseg > 1) the segmented search: checks, norms, one candidate round (two for
// k > 33, the second admitting only keys beyond the first round's 32nd), finish.  The arguments are checked by the callers.
int knn_search(const float* X, int n, int d, int k, int row_begin, int row_end, const int* seg_ptr, int nseg, int* knn_idx,
               float* knn_dist, int* info, void* ws, size_t ws_bytes, cudaStream_t st) {
  KnnPlan p = knn_plan(n, d, row_begin, row_end, 0, seg_ptr, nseg);
  KnnBufs b;
  const size_t need = knn_bufs(ws, n, d, k, p, nullptr, &b);
  if (ws_bytes < need) {
    set_error("kNN workspace too small: %zu < %zu", ws_bytes, need);
    return GLL_ERR_WORKSPACE;
  }
  GLL_REQUIRE(k <= KC + 1 || p.tc.ok, "k > 33 needs the tensor-core path (n >= 256, row range starting on a multiple of 128)");
  const char* sh = getenv("GLL_B200_KNN_SHARE");  // "0": every candidate set keeps its own threshold (experiments)
  if (sh && sh[0] == '0') b.thr_g = nullptr;
  SegDev sd;
  memset(&sd, 0, sizeof(sd));
  const SegDev* seg = nullptr;
  GLL_CUDA_CHECK(cudaMemsetAsync(b.small, 0, 256, st));
  if (b.win) {
    {
      GLL_PROF(KID_KNN_SEGMENTS, st);
      for (size_t o = 0; o < p.ints.size(); o += UPLOAD_INTS) {
        IntChunk c;
        const int cnt = (int)std::min<size_t>(UPLOAD_INTS, p.ints.size() - o);
        memcpy(c.v, p.ints.data() + o, sizeof(int) * (size_t)cnt);
        upload_ints_kernel<<<1, 256, 0, st>>>(c, cnt, b.ints + o);
      }
      seg_windows_kernel<<<nseg, 256, 0, st>>>(b.ints, b.win);
      GLL_LAUNCH_CHECK();
    }
    if (p.tc.ok) {
      sd.win = b.win;
      sd.gfirst = b.ints + nseg + 1;
      sd.gct = sd.gfirst + p.tc.row_tiles + 1;
      sd.bstart = sd.gct + p.tc.row_tiles;
      p.lay.gfirst = sd.gfirst;
      seg = &sd;
    }
  }
  int rc = launch_norms(X, n, d, p.tc, b, st);
  if (rc) return rc;
  if (k > KC + 1) {
    const int rows = row_end - row_begin;
    for (int round = 0; round < 2; ++round) {
      rc = knn_tc_candidates(X, b.sq, b.rscale, b.small, n, d, row_end, p.tc, b.tc_ws, b.cand, round ? b.excl : nullptr,
                             round ? nullptr : b.thr_g, st, seg);  // the second round keeps its own thresholds
      if (rc) return rc;
      {
        GLL_PROF(KID_RERANK, st);
        knn_merge_kernel<<<ceil_div(rows, RERANK_WARPS), RERANK_WARPS * 32, 0, st>>>(row_end, p.lay, b.cand,
                                                                                    b.merged + (size_t)round * rows * KC,
                                                                                    round ? nullptr : b.excl);
      }
      GLL_LAUNCH_CHECK();
    }
  } else if (p.tc.ok) {  // tcgen05 / TMA Gram GEMM with the fused top-k epilogue
    rc = knn_tc_candidates(X, b.sq, b.rscale, b.small, n, d, row_end, p.tc, b.tc_ws, b.cand, nullptr, b.thr_g, st, seg);
  } else {  // fp32 SIMT Gram (tiny graphs, or forced by GLL_B200_KNN_PATH=simt)
    rc = launch_simt(X, b.sq, n, d, p.cps, p.lay.stride, b.cand, row_begin, row_end, b.win, st);
  }
  if (rc) return rc;
  return knn_finish(X, n, d, k, row_end, p.lay, b.cand, p.err_coef, b, knn_idx, knn_dist, info, st);
}

}  // namespace

size_t knn_ws_bytes(int n, int d, int k, int row_begin, int row_end) {
  return knn_bufs(nullptr, n, d, k, knn_plan(n, d, row_begin, row_end), nullptr, nullptr);
}

int knn_run(const float* X, int n, int d, int k, int row_begin, int row_end, int* knn_idx, float* knn_dist, int* info,
            void* ws, size_t ws_bytes, cudaStream_t st) {
  GLL_REQUIRE(X && knn_idx && knn_dist && ws, "null pointer");
  GLL_REQUIRE(n >= k && k >= 2 && k <= 2 * KC, "need n >= k and 2 <= k <= 64");
  GLL_REQUIRE(d >= 1, "d must be positive");
  GLL_REQUIRE(0 <= row_begin && row_begin < row_end && row_end <= n, "bad row range");
  return knn_search(X, n, d, k, row_begin, row_end, nullptr, 1, knn_idx, knn_dist, info, ws, ws_bytes, st);
}

int knn_seg_check(int n, int d, int k, const int* seg_ptr, int nseg) {
  GLL_REQUIRE(seg_ptr != nullptr, "null seg_ptr");
  GLL_REQUIRE(nseg >= 1 && n >= 1 && d >= 1, "bad sizes");
  GLL_REQUIRE(k >= 2 && k <= 2 * KC && (k <= KC + 1 || n >= 2 * 128), "need 2 <= k <= 64, and n >= 256 when k > 33");
  GLL_REQUIRE(seg_ptr[0] == 0 && seg_ptr[nseg] == n, "seg_ptr must run from 0 to n");
  for (int s = 0; s < nseg; ++s)
    if (seg_ptr[s + 1] - seg_ptr[s] < k) {
      set_error("segment %d has %d rows, fewer than k = %d (or seg_ptr is not increasing)", s, seg_ptr[s + 1] - seg_ptr[s], k);
      return GLL_ERR_ARG;
    }
  return GLL_OK;
}

size_t knn_seg_ws_bytes(int n, int d, int k, const int* seg_ptr, int nseg) {
  if (knn_seg_check(n, d, k, seg_ptr, nseg) != GLL_OK) return 0;
  return knn_bufs(nullptr, n, d, k, knn_plan(n, d, 0, n, 0, seg_ptr, nseg), nullptr, nullptr);
}

// nseg == 1 is the plain search over all rows
int knn_run_segments(const float* X, int n, int d, int k, const int* seg_ptr, int nseg, int* knn_idx, float* knn_dist, int* info,
                     void* ws, size_t ws_bytes, cudaStream_t st) {
  GLL_REQUIRE(X && knn_idx && knn_dist && ws, "null pointer");
  const int rc = knn_seg_check(n, d, k, seg_ptr, nseg);
  if (rc) return rc;
  return knn_search(X, n, d, k, 0, n, seg_ptr, nseg, knn_idx, knn_dist, info, ws, ws_bytes, st);
}

// units the tensor-core search of a segmented call issues, and those of the uniform grid over the same rows (0, 0: SIMT path)
void knn_seg_units(int n, int d, const int* seg_ptr, int nseg, long long* seg_units, long long* uniform_units) {
  *seg_units = *uniform_units = 0;
  if (knn_seg_check(n, d, 2, seg_ptr, nseg) != GLL_OK) return;
  const TcPlan u = knn_tc_plan(n, d, 0, n);
  if (!u.ok) return;
  *uniform_units = u.units;
  if (nseg == 1) {
    *seg_units = u.units;
    return;
  }
  std::vector<int> tab;
  *seg_units = knn_tc_plan_segments(n, d, seg_ptr, nseg, &tab).units;
}

// Verification entry (gll_debug_gram_tile): operand split of the whole matrix as knn_run does it, then the raw tensor-core
// accumulator of unit (row_tile, col_tile) and the rows' operand scale 2^E_i.
int knn_debug_gram_tile(const float* X, int n, int d, int row_tile, int col_tile, float* acc_out, float* rscale_out, void* ws,
                        size_t ws_bytes, cudaStream_t st) {
  GLL_REQUIRE(X && acc_out && rscale_out && ws, "null pointer");
  GLL_REQUIRE(n >= 256 && d >= 1, "the tensor-core path needs n >= 256");
  const KnnPlan p = knn_plan(n, d, 0, n);
  KnnBufs b;
  const size_t need = knn_bufs(ws, n, d, 2, p, nullptr, &b);
  if (ws_bytes < need) {
    set_error("workspace too small: %zu < %zu", ws_bytes, need);
    return GLL_ERR_WORKSPACE;
  }
  GLL_REQUIRE(p.tc.ok, "tensor-core plan not available for this shape");
  GLL_REQUIRE(row_tile >= 0 && row_tile * 128 < n && col_tile >= 0 && col_tile * 256 < n, "tile out of range");
  GLL_CUDA_CHECK(cudaMemsetAsync(b.small, 0, 256, st));
  const int rcs = launch_norms(X, n, d, p.tc, b, st);
  if (rcs) return rcs;
  GLL_CUDA_CHECK(cudaMemcpyAsync(rscale_out, b.rscale, sizeof(float) * (size_t)n, cudaMemcpyDeviceToDevice, st));
  return knn_tc_debug_tile(p.tc, n, b.tc_ws, row_tile, col_tile, acc_out, st);
}

// ------------------------------------------------------------------------------------------------------------------------
// Base-set reuse across evaluation batches (SURVEY 8f-4; utils.py:596-621: test_network calls the layer on
// [base; test batch] with the SAME base rows for every batch).  The base-base part of the search -- n_base^2 of the
// (n_base + m)^2 pairs -- is done once: per base row the 32 best base columns (approximate keys, as the Gram kernel
// selects them).  Per call only the batch rows are searched against all columns and the base rows against the batch
// columns, each base row starting from its cached threshold; the merged candidates go through the usual exact re-rank
// and completeness proof (approximate distances only have to satisfy the error bound, whichever launch produced them),
// so the lists are the ones gll_knn gives on the concatenated matrix.
// ------------------------------------------------------------------------------------------------------------------------
namespace {

__global__ void base_thr_init_kernel(const u64* __restrict__ cache, const float* __restrict__ sq, const unsigned* __restrict__ small, int rows,
                                     unsigned* __restrict__ thr_g) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows) return;
  const u64 last = cache[(size_t)i * KC + KC - 1];
  float thr = INFINITY;
  if (last != KEY_INF) {
    // the epilogue compares d~^2 - |x_i|^2 with the threshold; the cached key holds fl(d~^2): undo the addition rounding UP
    // (a looser threshold only admits a few more candidates)
    // ... and the roundings of the epilogue's own arithmetic on shifted values (knn_tc.cu: a few ulps of max|x|^2)
    thr = __fadd_ru(key_dist(last), -sq[i]);
    thr = fmaf(fabsf(thr), 4.0e-7f, thr) + 2.0e-6f * __uint_as_float(small[0]) + 1.0e-30f;
  }
  thr_g[i] = float_to_ordered(thr);
}

// rows < r0: cached base list + the sets of the base x batch-columns launch; rows >= r0: the sets of the full-row launch
__global__ void __launch_bounds__(RERANK_WARPS * 32)
knn_merge_cached_kernel(int r0, int n, CandLayout layA, const u64* __restrict__ candA, CandLayout layB, const u64* __restrict__ candB,
                        const u64* __restrict__ cache, u64* __restrict__ merged) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.x * RERANK_WARPS + warp;
  if (i >= n) return;
  const bool base = i < r0;
  const CandLayout& lay = base ? layB : layA;
  const u64* cand = base ? candB : candA;
  u64 mine = base ? cache[(size_t)i * KC + lane] : KEY_INF;
  const int splits = cand_lists(lay, i);
  for (int s = 0; s < splits; ++s) list_merge_set(mine, cand[((size_t)i * lay.stride + s) * KC + lane], lane);
  merged[(size_t)i * KC + lane] = mine;
}

// The plans and the workspace of a cached search: batch rows [r0, n) against all columns, base rows [0, r0) against the batch
// columns.  One candidate round whatever k: the cached search serves k <= 33.
size_t cached_bufs(void* ws, int n, int d, int nb, KnnPlan* pa, KnnPlan* pb, KnnBufs* b) {
  const int r0 = nb / 128 * 128;  // base rows [r0, n_base) ride along with the batch rows (row ranges start on a tile)
  *pa = knn_plan(n, d, r0, n);
  *pb = knn_plan(n, d, 0, r0 > 0 ? r0 : 128, nb);
  return knn_bufs(ws, n, d, KC + 1, *pa, pb, b);
}

}  // namespace

size_t knn_base_cache_bytes(int n_base) { return align_up(sizeof(u64) * (size_t)n_base * KC, 256); }

// sized like gll_knn on the base rows (gll_base_cache_workspace_bytes)
int knn_base_cache_build(const float* Xb, int nb, int d, void* cache, void* ws, size_t ws_bytes, cudaStream_t st) {
  GLL_REQUIRE(Xb && cache && ws, "null pointer");
  GLL_REQUIRE(nb >= KC + 1 && d >= 1, "bad sizes");
  const KnnPlan p = knn_plan(nb, d, 0, nb);
  KnnBufs b;
  const size_t need = knn_bufs(ws, nb, d, 2, p, nullptr, &b);
  if (ws_bytes < need) {
    set_error("kNN workspace too small: %zu < %zu", ws_bytes, need);
    return GLL_ERR_WORKSPACE;
  }
  GLL_REQUIRE(p.tc.ok, "the base-set cache needs the tensor-core search (n_base >= 256)");
  GLL_CUDA_CHECK(cudaMemsetAsync(b.small, 0, 256, st));
  int rc = launch_norms(Xb, nb, d, p.tc, b, st);
  if (rc) return rc;
  rc = knn_tc_candidates(Xb, b.sq, b.rscale, b.small, nb, d, nb, p.tc, b.tc_ws, b.cand, nullptr, b.thr_g, st);
  if (rc) return rc;
  {
    GLL_PROF(KID_RERANK, st);
    knn_merge_kernel<<<ceil_div(nb, RERANK_WARPS), RERANK_WARPS * 32, 0, st>>>(nb, p.lay, b.cand, (u64*)cache, nullptr);
  }
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

size_t knn_cached_ws_bytes(int n, int d, int k, int nb) {
  (void)k;
  KnnPlan pa, pb;
  return cached_bufs(nullptr, n, d, nb, &pa, &pb, nullptr);
}

int knn_run_cached(const float* X, int n, int d, int k, int nb, const void* cache_v, int* knn_idx, float* knn_dist, int* info, void* ws,
                   size_t ws_bytes, cudaStream_t st) {
  GLL_REQUIRE(X && cache_v && knn_idx && knn_dist && ws, "null pointer");
  GLL_REQUIRE(k >= 2 && k <= KC + 1, "the base-set cache serves k <= 33");
  GLL_REQUIRE(nb >= KC + 1 && nb < n && d >= 1, "need 32 < n_base < n");
  KnnPlan pa, pb;
  KnnBufs b;
  const size_t need = cached_bufs(ws, n, d, nb, &pa, &pb, &b);
  if (ws_bytes < need) {
    set_error("kNN workspace too small: %zu < %zu", ws_bytes, need);
    return GLL_ERR_WORKSPACE;
  }
  const u64* cache = (const u64*)cache_v;
  const int r0 = pa.row_begin;
  GLL_REQUIRE(pa.tc.ok, "tensor-core plan not available for this shape");
  GLL_REQUIRE(r0 == 0 || pb.tc.ok, "tensor-core plan not available for this shape");
  GLL_CUDA_CHECK(cudaMemsetAsync(b.small, 0, 256, st));
  int rc;
  {
    GLL_PROF(KID_SQNORM, st);
    rc = launch_split_f16(X, n, d, pa.tc, b.sq, b.small, b.tc_ws, b.rscale, b.thr_g, st);
    if (rc) return rc;
    if (r0 > 0) base_thr_init_kernel<<<ceil_div(r0, 256), 256, 0, st>>>(cache, b.sq, b.small, r0, b.thr_g);
    GLL_LAUNCH_CHECK();
  }
  rc = knn_tc_candidates(X, b.sq, b.rscale, b.small, n, d, n, pa.tc, b.tc_ws, b.cand, nullptr, b.thr_g, st);
  if (rc) return rc;
  if (r0 > 0) {
    rc = knn_tc_candidates(X, b.sq, b.rscale, b.small, n, d, r0, pb.tc, b.tc_ws, b.cand_base, nullptr, b.thr_g, st);
    if (rc) return rc;
  }
  {
    GLL_PROF(KID_RERANK, st);
    knn_merge_cached_kernel<<<ceil_div(n, RERANK_WARPS), RERANK_WARPS * 32, 0, st>>>(r0, n, pa.lay, b.cand, pb.lay, b.cand_base,
                                                                                   cache, b.merged);
  }
  GLL_LAUNCH_CHECK();
  CandLayout one_list{};  // one sorted list per row
  one_list.stride = 1;
  return knn_finish(X, n, d, k, n, one_list, b.merged, pa.err_coef, b, knn_idx, knn_dist, info, st);
}

}  // namespace gll
