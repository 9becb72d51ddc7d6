// K1, tensor-core variant -- the pairwise-distance contraction behind knnsearch (GLL.py:181-189) as a tcgen05 / TMA GEMM
// with the per-row top-32 selection fused into the epilogue; the n x n matrix never leaves the SM.
//
// Arithmetic.  The GEMM only SELECTS 32 candidates per row; knn_rerank (knn.cu) recomputes them exactly in fp64, proves
// that no true neighbour was missed and redoes unprovable rows by brute force, so the emitted neighbour lists do not
// depend on tensor-core rounding.  Every row is scaled by an exact power of two to a norm in [148, 296) (no fp16
// overflow for any feature scale; rows normalised to 1 -- every caller of the layer -- all get the same scale) and
// rounded to fp16: z = hi (+ lo).  Default, ONE pass: Gram = hi_i . hi_j.  Its error is bounded rigorously by the measured
// operand residual rho = max_j |x_j - hi_j 2^E_j|_2 (~0.3 * 2^-11 |x_j|, exact in fp64, computed by the split kernel):
// |x_i.x_j - hi_i.hi_j| <= rho (|x_i| + |x_j| + rho), which for unit rows is 5.6e-4 in d^2 -- the same size as the fp32
// accumulation budget (with its 4x margin) that the proof carries anyway, and well below the 24th -> 32nd neighbour gaps
// (3e-3 .. 9e-3 at C2).  GLL_B200_KNN_SPLIT=f16x2: Gram = (hi_i + lo_i) . hi_j in TWO passes (A side exact to 2^-22, the
// bound keeps the one-sided 2 |x_i| rho): twice the MMA work for a bound that is 30 % tighter; kept for data whose neighbour
// gaps sit between the two bounds.  (Round 1's three-pass bf16 split is gone: same lists, 50 % more MMAs.)
//
// Kernel (one persistent CTA per SM, 11 warps, warp-specialised; every issue loop is run by a CONVERGED warp with
// warp-uniform operands and elect.sync around the issue itself, see elect_one()):
//   warp 0   TMA producer of the A operand: per 64-wide K block A_hi (128 rows, 16 KB; two passes: + A_lo), 128-byte swizzle
//   warp 10  TMA producer of the B operand: B_hi (256 rows, 32 KB; a CTA of a pair stages its half) into the same stage
//   warp 1   MMA issuer: 4 (two passes: 8) tcgen05.mma of K = 16 per stage into one of two 128 x 256 fp32 accumulators in
//            TMEM (all 512 columns; double buffered against the epilogue)
//   warps 2-9 epilogue, two per SM sub-partition: warps w and w+4 read the same TMEM lane quarter (the same 32 rows) and
//            take one half of the unit's 256 columns each.  tcgen05.ld gives each thread ONE row, 32 columns at a time;
//            v' = |xj|^2 + Cs - 2 acc (times the rows' scales) is compared with the row's threshold (a register): one
//            min per element and one vote decide whether the chunk holds any survivor at all.  A thread owns its row's
//            candidate set for its column half: an unsorted 32-slot array of packed (value | slot) keys in shared memory
//            (slot-major, so the 32 threads of a warp never bank-conflict), 4 groups of 8 slots whose largest keys are
//            cached in registers; a survivor replaces the overall maximum and only that group is rescanned.  All rows of a
//            warp insert concurrently.  The insertion is one long dependent chain (~75 instructions, ~430 cycles per round
//            of a warp), which is why a sub-partition gets two warps.  The warps never synchronise with each other.
//   thresholds  a row's sets (column halves, other CTAs on the same row tile) publish their 32nd-best through a per-row
//            word in L2 (atomicMin on the ordered-integer image of the float) and prune against each other's bound.
// Work = (row tile, column tile) units in row-major order, split evenly and contiguously over the CTAs, so a CTA keeps
// one row tile's sets on chip for many column tiles; sets are flushed to cand[row][slot][KC] when the row tile changes.
// PAIR: clusters of two CTAs on the same column tile, one tcgen05.mma.cta_group::2 of M = 256.
// What bounds it (tools/knn_trace.py; profiles/r02w_knn_trace_before.txt -> r02zd_knn_trace_after.txt): the EPILOGUE.  Reading a
// 128 x 256 fp32 accumulator out of TMEM takes ~2200 cycles (64 B per clock and SM) -- as long as its MMAs at d = 256 --
// plus the insertion rounds; the MMA/TMA pipeline alone runs a unit of d = 256 in ~3000 cycles (SS-mode operand reads from
// shared memory, not L2 bytes: a resident A operand changes nothing), the whole kernel in ~3800.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cudaTypedefs.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "knn_common.cuh"

namespace gll {
namespace {

// Stage = one 64-wide K block (128-byte swizzle): {A_hi 16 KB, B_hi 32 KB} for one pass, + A_lo 16 KB for two; a CTA of a
// pair stages half of B.  The ring takes all the shared memory the candidate sets of the EIGHT epilogue warps leave (152 KB:
// three 48 KB stages; five 16 KB B stages behind a resident 64 KB A operand at d = 256 with pairs).
constexpr int TC_BM = 128, TC_BN = 256, TC_BK = 64, TC_MAX_STAGES = 9;
constexpr size_t TC_STAGE_REGION = 152 * 1024;
// CTA pairs (cta_group::2, M = 256).  Measured (profiles/r02q_knn_experiments.txt): 4-7 % faster on the 1M-node graph (whole
// row tiles per CTA, drain-bound epilogue: fewer operand bytes and TMA issues per SM), no difference at 10-16 k nodes (bound
// by the candidate insertions).  Default: on from 8192 rows; GLL_B200_KNN_PAIR=0/1 forces it.
constexpr int TC_EPI_WARPS = 8;                        // two per TMEM lane quarter: each takes one half of the 256 columns
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS + 32;  // + the second TMA producer warp
constexpr int TC_WARP_PRODUCER_B = 2 + TC_EPI_WARPS;
constexpr int TC_A_BYTES = TC_BM * TC_BK * 2;          // 16 KB
constexpr int TC_B_BYTES = TC_BN * TC_BK * 2;          // 32 KB
constexpr int TC_STAGE_BYTES = 2 * TC_A_BYTES + TC_B_BYTES;  // 64 KB (the one-pass stage uses 48 KB)
constexpr int TC_CHUNK = 32;                           // columns per tcgen05.ld
constexpr int TC_TMEM_COLS = 512, TC_ACC_STRIDE = 256;

constexpr size_t TC_OFF_LD = TC_STAGE_REGION;                                // float [8 warps][KC entries][32 rows]
constexpr size_t TC_OFF_LI = TC_OFF_LD + TC_EPI_WARPS * KC * 32 * 4;         // int   [8 warps][KC entries][32 rows]
constexpr size_t TC_OFF_SQJ = TC_OFF_LI + TC_EPI_WARPS * KC * 32 * 4;        // float [8 warps][{|x_j|^2 + Cs, -2 rscale_j}][128 columns]
constexpr size_t TC_OFF_BAR = TC_OFF_SQJ + TC_EPI_WARPS * TC_BN * 4;         // mbarriers + tmem pointer
constexpr size_t TC_OFF_TMEM = TC_OFF_BAR + 8 * (2 * TC_MAX_STAGES + 6);     // the TMEM base address slot
constexpr size_t TC_SMEM_BYTES = TC_OFF_TMEM + 16 + 1024;                    // + slack for manual 1024 B alignment
static_assert(TC_SMEM_BYTES <= 227 * 1024, "shared memory budget");
static_assert(TC_STAGE_REGION / (2 * TC_A_BYTES) >= 1 && TC_STAGE_REGION % 1024 == 0, "stage ring");
static_assert(2 * TC_BN <= TC_TMEM_COLS && TC_ACC_STRIDE >= TC_BN, "two accumulators must fit in TMEM");

// M = 128, N = 256, A/B fp16 K-major (format fields 0), D fp32 (layout: cute::UMMA::InstrDescriptor)
constexpr uint32_t TC_IDESC_F16_PAIR = (1u << 4) | ((uint32_t)(TC_BN >> 3) << 17) | ((uint32_t)((2 * TC_BM) >> 4) << 24);  // M = 256
constexpr uint32_t TC_IDESC_F16 = (1u << 4) | ((uint32_t)(TC_BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);

// ---------------------------------------------------------------------------------------------- PTX wrappers
// One elected lane of a CONVERGED warp.  The TMA and MMA loops below are run by all 32 lanes with warp-uniform operands
// and only the issue itself sits under this predicate: operands then live in uniform registers.  Under `if (lane == 0)`
// the compiler treats them as per-thread values and wraps every UTMALDG / UTCHMMA into an ELECT + 5 x R2UR + branch
// "waterfall" (~170 cycles per tcgen05.mma, ~280 per cp.async.bulk.tensor: the MMA warp, not the tensor pipe or L2, paced
// the kernel -- tools/knn_trace.py, profiles/r02zc_mma_trace.txt).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as a trapped launch (error code), never as a hung GPU box.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  unsigned long long t0, t1;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (uint32_t spin = 1; !mbar_try_wait(bar, parity); ++spin) {
    if ((spin & 1023u) == 0) {
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > 4000000000ull) __trap();  // 4 s
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(x), "r"(y)
      : "memory");
}
// ---- CTA pair (cta_group::2): one tcgen05.mma of M = 256 spans two SMs of a TPC; each CTA holds its 128 rows of A and
// its 128 rows (= accumulator columns) of B in its own shared memory, the accumulator rows land in each CTA's own TMEM.
// Bit 24 of a shared-window address selects the CTA of the pair (cute: Sm100MmaPeerBitMask): cleared = the leader (rank 0).
constexpr uint32_t TC_PEER_MASK = 0xFEFFFFFFu;
// TMA load into MY shared memory whose completion bytes are counted by the LEADER's mbarrier
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar & TC_PEER_MASK), "r"(x), "r"(y)
      : "memory");
}
// arrive on the LEADER's mbarrier at this offset (from either CTA of the pair)
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & TC_PEER_MASK) : "memory");
}
__device__ __forceinline__ void tc_mma_f16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the barrier at the same offset in both CTAs once the pair's MMAs issued so far have retired
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// K-major operand tile whose rows are one swizzle atom wide (TC_BK fp16 = 64 B), 8-row groups 8 rows apart
// (cute::UMMA::SmemDescriptor; layout type 2 = SWIZZLE_128B, 4 = SWIZZLE_64B)
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t addr) {
  constexpr uint64_t sbo = (uint64_t)(8 * TC_BK * 2) >> 4, layout = (TC_BK == 64) ? 2 : 4;
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | (sbo << 32) | ((uint64_t)1 << 46) | (layout << 61);
}
// Asynchronous TMEM -> register load of 32 consecutive columns of this thread's row; the registers are valid only after
// tc_ld_wait(), which names them as in/out operands so that no use can be scheduled ahead of the wait.  (16-column loads
// left the epilogue latency-bound once the f16x2 split had shortened the MMA time per unit: one wait + one vote per chunk.)
#define TC_R8(o, b) o(r[b + 0]), o(r[b + 1]), o(r[b + 2]), o(r[b + 3]), o(r[b + 4]), o(r[b + 5]), o(r[b + 6]), o(r[b + 7])
#define TC_OUT(x) "=r"(x)
#define TC_INOUT(x) "+r"(x)
__device__ __forceinline__ void tc_ld_issue(uint32_t taddr, uint32_t (&r)[TC_CHUNK]) {
  static_assert(TC_CHUNK == 32, "the asm below names 32 registers");
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : TC_R8(TC_OUT, 0), TC_R8(TC_OUT, 8), TC_R8(TC_OUT, 16), TC_R8(TC_OUT, 24)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tc_ld_wait(uint32_t (&r)[TC_CHUNK]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : TC_R8(TC_INOUT, 0), TC_R8(TC_INOUT, 8), TC_R8(TC_INOUT, 16), TC_R8(TC_INOUT, 24)
               :
               : "memory");
}
#undef TC_R8
#undef TC_OUT
#undef TC_INOUT

struct TcParams {
  int n, kblocks, col_tiles, max_splits;
  int rt0, row_end;   // first row tile of this call's row range, one past its last row
  int ct0, col_begin; // first column tile / first column of this call's column range (columns before col_begin are masked)
  int aligned;        // 1: every CTA owns whole row tiles (all CTAs sweep the column tiles in lockstep: B tiles hit in L2)
  int row_tiles;
  long long units;
  const float* sq;
  u64* cand;
  unsigned* thr_g;    // [n] per-row threshold shared by every candidate set of the row (ordered-uint of the float), or NULL
  int debug;          // GLL_B200_KNN_DEBUG (timing experiments only, results are wrong): 1 no insertions, 2 no TMEM drain
  const u64* excl;    // optional [n]: per row, only keys > excl[row] are candidates (second round of a k > 33 search)
  int passes;         // operands are fp16(x_i 2^-E_i): 1 = hi.hi, 2 = (hi + lo).hi (B_lo never exists)
  int ares;           // 1: all K blocks of the row tile's A operand stay in shared memory while the CTA sweeps column tiles
  const float* rscale;  // [n] 2^E_i: the accumulator holds x_i.x_j / (rscale_i rscale_j)
  const unsigned* small;  // small[3], small[4]: range of E_i over the rows (written by sqnorm_split_f16_kernel)
  unsigned long long* trace;  // debug timeline of CTA 0 (gll_debug_knn_trace, tools/knn_trace.py), or NULL
};
constexpr int TC_TRACE_UNITS = 1024, TC_TRACE_PHASES = 8;  // four traced warps: MMA warp, epilogue warps 2 and 6, producer A

__host__ __device__ inline uint32_t a_bytes_of(int passes) { return passes == 2 ? 2u * TC_A_BYTES : (uint32_t)TC_A_BYTES; }  // A_hi (+ A_lo)

// CTA that owns unit u when `units` units are dealt contiguously to G CTAs (CTA b owns [b*units/G, (b+1)*units/G))
__host__ __device__ inline int tc_cta_of_unit(long long u, int G, long long units) { return (int)(((u + 1) * G - 1) / units); }

// Segmented unit grid: row group r's column-tile count and first column tile (r == row_tiles: past the end, left alone)
__device__ __forceinline__ void seg_group(const SegDev& S, int row_tiles, int r, int& cnt, int& ctl) {
  if (r < row_tiles) {
    cnt = __ldg(S.gfirst + r + 1) - __ldg(S.gfirst + r);
    ctl = __ldg(S.gct + r);
  }
}

// ---------------------------------------------------------------------------------------------- the GEMM + top-k kernel
// PAIR: launched as clusters of two CTAs (one TPC) that process the SAME column tile for two adjacent row tiles with ONE
// tcgen05.mma.cta_group::2 of M = 256: each CTA stages its own 128 rows of A and HALF of the B tile (128 of the 256
// columns), so the operand bytes a CTA pulls from L2 drop by a third -- which is what bounds the one-pass kernel
// (measured: ~70 GB/s per SM whatever the stage count, profiles/r02k_knn_experiments_c2.txt).  The leader CTA issues the
// MMAs; both CTAs run their own TMA producer and their own epilogue on their own 128 accumulator rows.
// SEG: segmented search.  Row group r_idx has cnt column tiles from ctl on (S); the uniform grid has cnt = C, ctl = ct0.  S is
// a parameter of its own: inside TcParams it would push the struct past the size up to which the compiler keeps it in registers.
template <bool PAIR, bool SEG>
__global__ void __launch_bounds__(TC_THREADS, 1)
knn_gram_topk_tc_kernel(const __grid_constant__ CUtensorMap mapAH, const __grid_constant__ CUtensorMap mapAL,
                        const __grid_constant__ CUtensorMap mapBH, TcParams P, SegDev S) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;  // 128B-swizzled operand tiles need 1024 B alignment
  uint8_t* smem = smem_raw + (base - raw);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // work is dealt to CTAs, or to CTA pairs: G owners, this CTA belongs to owner b and is rank `crank` inside it
  const int crank = PAIR ? (int)cluster_ctarank() : 0;
  const int G = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x, b = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int RSTEP = PAIR ? 2 : 1;  // row tiles per unit
  const int C = P.col_tiles, KB = P.kblocks;
  const bool tracing = P.trace != nullptr && blockIdx.x == 0 && lane == 0;
  auto stamp = [&](int w, long long ui, int ph, long long val) {
    if (tracing && ui < TC_TRACE_UNITS) P.trace[((size_t)w * TC_TRACE_UNITS + ui) * TC_TRACE_PHASES + ph] = (unsigned long long)val;
  };
  long long u_begin, u_end;
  // SEG: coordinates of unit u_begin (row-group ordinal, column-tile ordinal inside it, the group's tile count and first tile).
  // The uniform grid keeps its own arithmetic below, in each warp role, exactly as without segments.
  int r_begin = 0, c_begin0 = 0, cnt0 = C, ctl0 = P.ct0;
  if constexpr (SEG) {
    if (P.aligned) {
      const int g0 = (int)((long long)b * P.row_tiles / G), g1 = (int)((long long)(b + 1) * P.row_tiles / G);
      u_begin = (long long)__ldg(S.gfirst + g0);
      u_end = (long long)__ldg(S.gfirst + g1);
      r_begin = g0;
    } else {
      u_begin = (long long)b * P.units / G;
      u_end = (long long)(b + 1) * P.units / G;
      r_begin = __ldg(S.bstart + b);
    }
    seg_group(S, P.row_tiles, r_begin, cnt0, ctl0);
    c_begin0 = (r_begin < P.row_tiles) ? (int)(u_begin - __ldg(S.gfirst + r_begin)) : 0;
  } else {
    if (P.aligned) {
      u_begin = ((long long)b * P.row_tiles / G) * C;
      u_end = ((long long)(b + 1) * P.row_tiles / G) * C;
    } else {
      u_begin = (long long)b * P.units / G;
      u_end = (long long)(b + 1) * P.units / G;
    }
  }

  const bool two = P.passes == 2;
  const uint32_t a_bytes = two ? 2u * TC_A_BYTES : (uint32_t)TC_A_BYTES;  // A_hi (+ A_lo) of one K block
  const uint32_t b_bytes = (uint32_t)(PAIR ? TC_B_BYTES / 2 : TC_B_BYTES);  // what THIS CTA loads of a B tile's K block
  // ares (A resident): the KB blocks of the row tile's A operand sit at the start of the stage region for as long as the CTA
  // stays on the row tile and the ring only carries B -- on the 1M-node graph (4096 column tiles per row tile) this halves
  // the operand bytes a CTA pulls from L2, which is what paces the MMA/TMA pipeline there (~40 B per clock and SM).
  const bool ares = P.ares != 0;
  const uint32_t ring_base = base + (ares ? (uint32_t)KB * a_bytes : 0u);
  const uint32_t stage_stride = ares ? b_bytes : a_bytes + b_bytes;  // = bytes this CTA loads per stage
  const int nstages = min(TC_MAX_STAGES, (int)(((uint32_t)TC_STAGE_REGION - (ring_base - base)) / stage_stride));
  const uint32_t bar_full = base + (uint32_t)TC_OFF_BAR;        // [TC_MAX_STAGES]
  const uint32_t bar_empty = bar_full + 8 * TC_MAX_STAGES;      // [TC_MAX_STAGES]
  const uint32_t bar_tfull = bar_empty + 8 * TC_MAX_STAGES;     // [2]
  const uint32_t bar_tempty = bar_tfull + 16;                   // [2]
  const uint32_t bar_afull = bar_tempty + 16;                   // ares: the resident A operand has landed
  const uint32_t bar_afree = bar_afull + 8;                     // ares: every MMA that reads the resident A operand has retired
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + TC_OFF_TMEM);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapAH);
    tma_prefetch_desc(&mapAL);
    tma_prefetch_desc(&mapBH);
    for (int s = 0; s < TC_MAX_STAGES; ++s) {
      mbar_init(bar_full + 8 * s, ares ? 1 : 2);  // the two producer warps (ares: the B producer alone)
      mbar_init(bar_empty + 8 * s, 1);  // PAIR: the leader's commit arrives on both CTAs' barriers
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_tfull + 8 * a, 1);
      mbar_init(bar_tempty + 8 * a, PAIR ? 2 * TC_EPI_WARPS : TC_EPI_WARPS);  // one arrival per epilogue warp (PAIR: of both CTAs, on the leader)
    }
    mbar_init(bar_afull, 1);
    mbar_init(bar_afree, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (PAIR) {  // the same warp of both CTAs, the same destination offset
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(base + (uint32_t)TC_OFF_TMEM),
                   "r"((uint32_t)TC_TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(base + (uint32_t)TC_OFF_TMEM),
                   "r"((uint32_t)TC_TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if (PAIR)
    cluster_sync_all();  // the peer's barriers must exist before anything is multicast into this CTA
  else
    __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 || warp == TC_WARP_PRODUCER_B) {
    // ================================================= TMA producers ================================================
    // Warp 0 loads the A tiles, a second producer warp the B tile; both arrive on the stage's barrier with their own byte
    // counts.  (The split dates from the lane-0 issue form, where one cp.async.bulk.tensor cost its thread ~280 cycles.)
    if (ares && warp == 0) {
      // resident A: one load of all K blocks per row tile, after the MMAs of the previous row tile have retired
      int r_idx = SEG ? r_begin : (int)(u_begin / C), c_idx = SEG ? c_begin0 : (int)(u_begin % C);
      int cnt = cnt0, ctl = ctl0;  // SEG only
      (void)ctl;
      uint32_t ph_free = 0;
      for (long long u = u_begin; u < u_end;) {
        const int rt = P.rt0 + RSTEP * r_idx + crank;
        if (u != u_begin) {
          mbar_wait(bar_afree, ph_free);
          ph_free ^= 1u;
        }
        if (elect_one()) {
          if (PAIR) {  // both CTAs' loads are counted by the LEADER's barrier (its MMA warp is the only consumer)
            if (crank == 0) mbar_arrive_expect_tx(bar_afull, 2u * (uint32_t)KB * a_bytes);
            for (int kk = 0; kk < KB; ++kk) {
              tma_load_2d_pair(base + (uint32_t)kk * a_bytes, &mapAH, bar_afull, kk * TC_BK, rt * TC_BM);
              if (two) tma_load_2d_pair(base + (uint32_t)kk * a_bytes + TC_A_BYTES, &mapAL, bar_afull, kk * TC_BK, rt * TC_BM);
            }
          } else {
            mbar_arrive_expect_tx(bar_afull, (uint32_t)KB * a_bytes);
            for (int kk = 0; kk < KB; ++kk) {
              tma_load_2d(base + (uint32_t)kk * a_bytes, &mapAH, bar_afull, kk * TC_BK, rt * TC_BM);
              if (two) tma_load_2d(base + (uint32_t)kk * a_bytes + TC_A_BYTES, &mapAL, bar_afull, kk * TC_BK, rt * TC_BM);
            }
          }
        }
        __syncwarp();
        u += (SEG ? cnt : C) - c_idx;  // on to the CTA's next row tile
        c_idx = 0;
        ++r_idx;
        if constexpr (SEG) seg_group(S, P.row_tiles, r_idx, cnt, ctl);
      }
    } else {
      const bool is_a = warp == 0;
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t my_bytes = is_a ? a_bytes : b_bytes;
      const uint32_t b_off = ares ? 0u : a_bytes;  // where the B block sits inside a stage
      // the unit's row-tile ordinal and column tile, kept incrementally
      int r_idx = SEG ? r_begin : (int)(u_begin / C), c_idx = SEG ? c_begin0 : (int)(u_begin % C);
      int cnt = cnt0, ctl = ctl0;  // SEG only
      for (long long u = u_begin; u < u_end; ++u) {
        const int rt = P.rt0 + RSTEP * r_idx + crank, ct = (SEG ? ctl : P.ct0) + c_idx;
        if (++c_idx == (SEG ? cnt : C)) {
          c_idx = 0;
          ++r_idx;
          if constexpr (SEG) seg_group(S, P.row_tiles, r_idx, cnt, ctl);
        }
        if (is_a && tracing) stamp(3, u - u_begin, 0, clock64());
        for (int kk = 0; kk < KB; ++kk) {
          mbar_wait(bar_empty + 8 * stage, phase ^ 1u);
          if (is_a && tracing && kk == KB - 1) stamp(3, u - u_begin, 1, clock64());
          const uint32_t full = bar_full + 8 * stage;
          const uint32_t s0 = ring_base + (uint32_t)stage * stage_stride;
          if (elect_one()) {
            if (PAIR) {
              // both CTAs' loads of this stage are counted by the LEADER's barrier (its MMA warp is the only consumer)
              if (crank == 0) mbar_arrive_expect_tx(full, 2u * my_bytes);
              if (is_a) {
                tma_load_2d_pair(s0, &mapAH, full, kk * TC_BK, rt * TC_BM);
                if (two) tma_load_2d_pair(s0 + TC_A_BYTES, &mapAL, full, kk * TC_BK, rt * TC_BM);
              } else {  // my half of the B tile: 128 of its 256 rows (128-row boxes: the A map)
                tma_load_2d_pair(s0 + b_off, &mapAH, full, kk * TC_BK, ct * TC_BN + crank * (TC_BN / 2));
              }
            } else {
              mbar_arrive_expect_tx(full, my_bytes);
              if (is_a) {
                tma_load_2d(s0, &mapAH, full, kk * TC_BK, rt * TC_BM);
                if (two) tma_load_2d(s0 + TC_A_BYTES, &mapAL, full, kk * TC_BK, rt * TC_BM);
              } else {
                tma_load_2d(s0 + b_off, &mapBH, full, kk * TC_BK, ct * TC_BN);
              }
            }
          }
          __syncwarp();
          if (++stage == nstages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================= MMA issuer (PAIR: the leader CTA only) =========================
    int stage = 0, acc = 0;
    uint32_t phase = 0, acc_phase = 0;
    const int nprod = P.passes;
    const uint32_t idesc = PAIR ? TC_IDESC_F16_PAIR : TC_IDESC_F16;
    int c_idx = SEG ? c_begin0 : (int)(u_begin % C);
    int r_idx = r_begin, cnt = cnt0, ctl = ctl0;  // SEG only
    (void)ctl;
    uint32_t ph_afull = 0;
    bool need_a = ares;
    for (long long u = (PAIR && crank != 0) ? u_end : u_begin; u < u_end; ++u) {
      if (tracing) stamp(0, u - u_begin, 0, clock64());
      mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1u);  // the epilogue has drained this accumulator
      if (need_a) {  // first unit of a row tile: the resident A operand
        mbar_wait(bar_afull, ph_afull);
        ph_afull ^= 1u;
        need_a = false;
      }
      const bool row_done = (++c_idx == (SEG ? cnt : C));  // last unit of the row tile
      if (row_done) c_idx = 0;
      if constexpr (SEG) {
        if (row_done) seg_group(S, P.row_tiles, ++r_idx, cnt, ctl);
      }
      tc_fence_after();
      if (tracing) stamp(0, u - u_begin, 1, clock64());
      const uint32_t d_tmem = tmem_base + (uint32_t)acc * TC_ACC_STRIDE;
      for (int kk = 0; kk < KB; ++kk) {
        mbar_wait(bar_full + 8 * stage, phase);
        tc_fence_after();
        if (tracing && kk == 0) stamp(0, u - u_begin, 2, clock64());
        if (tracing && kk == KB - 1) stamp(0, u - u_begin, 3, clock64());
        if (tracing && kk == 1) stamp(0, u - u_begin, 4, clock64());
        if (tracing && kk == 2) stamp(0, u - u_begin, 5, clock64());
        const uint32_t s0 = ring_base + (uint32_t)stage * stage_stride;
        const uint32_t sa = ares ? base + (uint32_t)kk * a_bytes : s0;
        const uint64_t dAH = tc_smem_desc(sa), dAL = tc_smem_desc(sa + TC_A_BYTES);
        const uint64_t dBH = tc_smem_desc(ares ? s0 : s0 + a_bytes);
        if (elect_one()) {
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            if (g >= nprod) break;  // one pass: hi.hi only
            const uint64_t da = (g == 1) ? dAL : dAH, db = dBH;  // hi.hi, lo.hi
#pragma unroll
            for (int k4 = 0; k4 < TC_BK / 16; ++k4) {  // +32 B (two 16 B units) per K=16 step inside the swizzle atom
              if (PAIR)
                tc_mma_f16_pair(d_tmem, da + (uint64_t)(2 * k4), db + (uint64_t)(2 * k4), idesc, (uint32_t)((kk | g | k4) != 0));
              else
                tc_mma_f16(d_tmem, da + (uint64_t)(2 * k4), db + (uint64_t)(2 * k4), idesc, (uint32_t)((kk | g | k4) != 0));
            }
          }
          // the resident A operand may be overwritten once the row tile's last MMAs have retired (committed BEFORE the
          // accumulator: when the epilogue of the CTA's last unit is through, nothing is in flight towards the peer any more)
          const bool a_done = ares && row_done && kk == KB - 1 && u + 1 < u_end;
          if (PAIR) {
            tc_commit_pair(bar_empty + 8 * stage);                 // frees the stage in BOTH CTAs when these MMAs retire
            if (a_done) tc_commit_pair(bar_afree);
            if (kk == KB - 1) tc_commit_pair(bar_tfull + 8 * acc);  // accumulator complete, in both CTAs' TMEM
          } else {
            tc_commit(bar_empty + 8 * stage);      // frees the smem stage when these MMAs retire
            if (a_done) tc_commit(bar_afree);
            if (kk == KB - 1) tc_commit(bar_tfull + 8 * acc);  // accumulator complete
          }
        }
        __syncwarp();
        if (tracing && kk == 0) stamp(0, u - u_begin, 6, clock64());        // the first K block's MMAs and commit are issued
        if (tracing && kk == KB - 1) stamp(0, u - u_begin, 7, clock64());   // ... and the last one's
        if (++stage == nstages) {
          stage = 0;
          phase ^= 1u;
        }
      }
      if (row_done) need_a = ares;
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1u;
    }
  } else {
    // ================================================= epilogue =====================================================
    // Every SM sub-partition hosts TWO epilogue warps (w and w + 4: same TMEM lane quarter, i.e. the same 32 rows); each
    // scans one half of the unit's 256 columns into its OWN candidate set, so a row has two sets per CTA.  The warps are
    // independent of each other: each stages the column norms of its own 128 columns (no CTA-wide barrier), so a warp that
    // runs insertion rounds delays nobody but itself, and only through the accumulator hand-off (tools/knn_trace.py: with a
    // barrier per unit every round of any warp cost all eight ~600 cycles).
    const int quarter = warp & 3;          // TMEM lanes [32*quarter, +32) are the ones this warp may read
    const int half = (warp - 2) >> 2;      // which 128 columns of the unit
    const int eset = half * 4 + quarter;   // the warp's block of candidate sets
    // A row's set: 32 slots of PACKED keys = (bits of the shifted value v' with the low five mantissa bits cleared) | slot, and
    // the column index beside it.  v' = d~^2 - |x_i|^2 + Cs with Cs = 2 max|x|^2 is positive, so unsigned order of the keys =
    // order of the values, ties by slot: ONE integer max finds the largest entry AND where it sits.  Clearing five bits costs
    // nothing in rigour: every threshold is a stored (cleared) value, a rejected column has v' >= threshold >= the final set
    // maximum as stored, and the stored values are what goes to the re-rank kernel (whose proof only needs "every column
    // that is not a candidate has an approximate distance >= the 32nd candidate's").
    uint32_t* Lk = reinterpret_cast<uint32_t*>(smem + TC_OFF_LD) + (size_t)eset * KC * 32 + lane;  // my row: Lk[e * 32]
    int* Li = reinterpret_cast<int*>(smem + TC_OFF_LI) + (size_t)eset * KC * 32 + lane;
    constexpr uint32_t KEY_EMPTY = 0x7f800000u;  // +inf
    int acc = 0, cur_rt = -1, gi = 0;
    uint32_t gk[4];  // largest key of slots [8t, 8t+8) of my row's set
    uint32_t acc_phase = 0;
    // thr = min(smax, tlim): smax = largest entry of MY set (inf until it is full), tlim = what the row's other sets --
    // the partner warp's column half, other CTAs working on the same row tile -- have published through thr_g (L2).
    // Any set's 32nd-best bounds the row's overall 32nd-best from above, so entries >= tlim can never be needed; the
    // union of the row's sets still holds the overall 32 best, and sets fill far more slowly (fewer insertions).
    float thr = INFINITY, smax = INFINITY, tlim = INFINITY, published = INFINITY;
    bool fresh_set = false;  // the set is empty: the first 32 columns go straight into the 32 slots
    u64 excl_row = 0ull;   // second-round searches: skip everything the first round already holds
    float sqi_row = 0.f;
    // this warp's staging area: |x_j|^2 + Cs of its 128 columns, then -2 rscale_j
    float* sq_w = reinterpret_cast<float*>(smem + TC_OFF_SQJ) + (size_t)(warp - 2) * TC_BN;
    float* cj_w = sq_w + TC_BN / 2;
    // d~^2 - |x_i|^2 = |x_j|^2 + (acc ri) cj with cj = -2 rscale_j, ri = rscale_i (powers of two: exact; 1 without scaling)
    float ri = 1.f;
    // all rows share one scale (the usual case: normalised features; always without scaling): v = |x_j|^2 + cu acc
    bool uniform = true;
    float cu = -2.f;
    if (P.rscale != nullptr) {
      const unsigned emax = __ldg(P.small + 3), eminc = __ldg(P.small + 4);  // biased max E, 255 - biased min E (knn.cu)
      uniform = (emax == 255u - eminc);
      cu = -ldexpf(2.f, 2 * ((int)emax - 128));
    }
    const float Cs = 2.f * __uint_as_float(__ldg(P.small + 0));  // v + Cs >= max|x|^2 - (error bound) > 0
    // value that goes to the candidate lists: fl(fl(v' - Cs) + |x_i|^2), monotone in v'
    auto unshift = [&](float vs, float sqr) { return (vs - Cs) + sqr; };

    auto flush = [&](int rt) {
      __syncwarp();
      int slot;
      if constexpr (SEG)
        slot = 2 * (P.aligned ? 0 : b - tc_cta_of_unit(__ldg(S.gfirst + (rt - P.rt0) / RSTEP), G, P.units)) + half;
      else
        slot = 2 * (P.aligned ? 0 : b - tc_cta_of_unit((long long)((rt - P.rt0) / RSTEP) * C, G, P.units)) + half;
      const uint32_t* wk = Lk - lane;
      const int* wi = Li - lane;
      for (int r = 0; r < 32; ++r) {  // lane = slot index e here; 256 B coalesced store per row
        const int row = rt * TC_BM + quarter * 32 + r;
        const uint32_t kk = wk[lane * 32 + r];
        const float sqr = (row < P.n) ? __ldg(P.sq + row) : 0.f;
        const u64 key = (kk >= KEY_EMPTY) ? KEY_INF : make_key(unshift(__uint_as_float(kk & ~31u), sqr), wi[lane * 32 + r]);
        if (row < P.row_end) P.cand[((size_t)row * P.max_splits + slot) * KC + lane] = key;
      }
      __syncwarp();
    };

    // |x_j|^2 + Cs (and -2 rscale_j) of my four columns of a unit, +inf masking columns outside the column range.  The values
    // of unit u + 1 are fetched into registers at the top of unit u and staged at the top of unit u + 1: their L2 round trip
    // is never in the epilogue's critical path (the kernel is bound by the epilogue).
    const int mycol = half * (TC_BN / 2) + 4 * lane;
    auto col_sq = [&](int ctile) {
      const int j = ctile * TC_BN + mycol;
      float4 r;
      r.x = (j + 0 < P.n && j + 0 >= P.col_begin) ? __ldg(P.sq + j + 0) : INFINITY;  // (Cs is added when the values are staged:
      r.y = (j + 1 < P.n && j + 1 >= P.col_begin) ? __ldg(P.sq + j + 1) : INFINITY;  //  nothing here may wait for the loads)
      r.z = (j + 2 < P.n && j + 2 >= P.col_begin) ? __ldg(P.sq + j + 2) : INFINITY;
      r.w = (j + 3 < P.n && j + 3 >= P.col_begin) ? __ldg(P.sq + j + 3) : INFINITY;
      return r;
    };
    auto col_cj = [&](int ctile) {
      const int j = ctile * TC_BN + mycol;
      float4 r;
      r.x = (j + 0 < P.n) ? __ldg(P.rscale + j + 0) : 1.f;  // (times -2 when staged)
      r.y = (j + 1 < P.n) ? __ldg(P.rscale + j + 1) : 1.f;
      r.z = (j + 2 < P.n) ? __ldg(P.rscale + j + 2) : 1.f;
      r.w = (j + 3 < P.n) ? __ldg(P.rscale + j + 3) : 1.f;
      return r;
    };
    // kept incrementally: no 64-bit divisions per unit
    int r_idx = SEG ? r_begin : (int)(u_begin / C), c_idx = SEG ? c_begin0 : (int)(u_begin % C);
    int cnt = cnt0, ctl = ctl0;  // SEG only
    // SEG: my row's column window [my_lo, my_hi), and the part [w_lo, w_hi) that every row of the warp shares
    int my_lo = 0, my_hi = 0, w_lo = 0, w_hi = 0;
    float4 nsq = make_float4(0.f, 0.f, 0.f, 0.f), ncj = nsq;
    if (u_begin < u_end) {
      nsq = col_sq((SEG ? ctl : P.ct0) + c_idx);
      if (!uniform) ncj = col_cj((SEG ? ctl : P.ct0) + c_idx);
    }
    for (long long u = u_begin; u < u_end; ++u) {
      const int rt = P.rt0 + RSTEP * r_idx + crank, ct = (SEG ? ctl : P.ct0) + c_idx;
      if (++c_idx == (SEG ? cnt : C)) {
        c_idx = 0;
        ++r_idx;
        if constexpr (SEG) seg_group(S, P.row_tiles, r_idx, cnt, ctl);
      }
      if (rt != cur_rt) {
        if (cur_rt >= 0) flush(cur_rt);
#pragma unroll
        for (int e = 0; e < KC; ++e) Lk[e * 32] = KEY_EMPTY | (uint32_t)e;
        cur_rt = rt;
        thr = smax = tlim = published = INFINITY;
        fresh_set = (P.excl == nullptr);
#pragma unroll
        for (int t = 0; t < 4; ++t) gk[t] = KEY_EMPTY | (uint32_t)(8 * t + 7);
        gi = rt * TC_BM + quarter * 32 + lane;
        ri = (P.rscale != nullptr && gi < P.n) ? __ldg(P.rscale + gi) : 1.f;
        if (P.excl != nullptr) {
          excl_row = (gi < P.n) ? __ldg(P.excl + gi) : 0ull;
          sqi_row = (gi < P.n) ? __ldg(P.sq + gi) : 0.f;
        }
        if constexpr (SEG) {  // rows past n see every column; their sets are never flushed
          const int2 w = (gi < P.n) ? __ldg(S.win + gi) : make_int2(0, 0x7fffffff);
          my_lo = w.x;
          my_hi = w.y;
          w_lo = __reduce_max_sync(FULL, my_lo);
          w_hi = __reduce_min_sync(FULL, my_hi);
        }
      }
      const int c_begin = ct * TC_BN;
      const int tw = !tracing ? -1 : (warp == 2) ? 1 : (warp == 6) ? 2 : -1;  // (tracing: lane 0 of CTA 0, debug runs only)
      int nround = 0;
      if (tw > 0) stamp(tw, u - u_begin, 0, clock64());
      if (tw == 1 && ((u - u_begin) & 1023) == 0) {  // coarse timeline of the whole CTA: SM clock and wall clock every 1024 units
        unsigned long long gt;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        stamp(1, (u - u_begin) >> 10, 6, (long long)gt);
        stamp(1, (u - u_begin) >> 10, 7, clock64());
      }
      // stage this unit's column values (fetched one unit ago), then put the next unit's in flight
      __syncwarp();  // every lane is done with the previous unit's values
      *reinterpret_cast<float4*>(sq_w + 4 * lane) = make_float4(nsq.x + Cs, nsq.y + Cs, nsq.z + Cs, nsq.w + Cs);
      if (!uniform) *reinterpret_cast<float4*>(cj_w + 4 * lane) = make_float4(-2.f * ncj.x, -2.f * ncj.y, -2.f * ncj.z, -2.f * ncj.w);
      __syncwarp();
      if (u + 1 < u_end) {
        nsq = col_sq((SEG ? ctl : P.ct0) + c_idx);
        if (!uniform) ncj = col_cj((SEG ? ctl : P.ct0) + c_idx);
      }
      // ... and what the row's other sets have published (once per unit; folded in after the first 32 columns, when the
      // load has landed)
      unsigned tg = 0xffffffffu;
      if (P.thr_g != nullptr && gi < P.n) tg = __ldcg(P.thr_g + gi);
      if (tw > 0) stamp(tw, u - u_begin, 1, clock64());
      // does this warp's row range meet this unit's column range?  (only then can a column be the row itself)
      const int wrow0 = rt * TC_BM + quarter * 32;
      const bool diag = (c_begin < wrow0 + 32) && (c_begin + TC_BN > wrow0);

      if (tw > 0) stamp(tw, u - u_begin, 2, clock64());
      mbar_wait(bar_tfull + 8 * acc, acc_phase);
      tc_fence_after();
      if (tw > 0) stamp(tw, u - u_begin, 3, clock64());
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)acc * TC_ACC_STRIDE;
      uint32_t rawA[TC_CHUNK], rawB[TC_CHUNK];
      // qq = chunk of this warp's column half (0..3)
      auto process = [&](const uint32_t (&raw)[TC_CHUNK], int qq) {
        const int j0 = c_begin + half * (TC_BN / 2) + qq * TC_CHUNK;
        float v[TC_CHUNK];
        uint32_t hits = 0;
        if (uniform) {  // every row has the same scale: one FMA per element (same value, the factors are powers of two)
#pragma unroll
          for (int c4 = 0; c4 < TC_CHUNK / 4; ++c4) {
            const float4 s4 = *reinterpret_cast<const float4*>(sq_w + qq * TC_CHUNK + 4 * c4);  // warp-wide broadcast
            v[4 * c4 + 0] = fmaf(__uint_as_float(raw[4 * c4 + 0]), cu, s4.x);
            v[4 * c4 + 1] = fmaf(__uint_as_float(raw[4 * c4 + 1]), cu, s4.y);
            v[4 * c4 + 2] = fmaf(__uint_as_float(raw[4 * c4 + 2]), cu, s4.z);
            v[4 * c4 + 3] = fmaf(__uint_as_float(raw[4 * c4 + 3]), cu, s4.w);
          }
        } else {
#pragma unroll
          for (int c4 = 0; c4 < TC_CHUNK / 4; ++c4) {
            const float4 s4 = *reinterpret_cast<const float4*>(sq_w + qq * TC_CHUNK + 4 * c4);  // warp-wide broadcast
            const float4 c4v = *reinterpret_cast<const float4*>(cj_w + qq * TC_CHUNK + 4 * c4);
            v[4 * c4 + 0] = fmaf(ri * __uint_as_float(raw[4 * c4 + 0]), c4v.x, s4.x);
            v[4 * c4 + 1] = fmaf(ri * __uint_as_float(raw[4 * c4 + 1]), c4v.y, s4.y);
            v[4 * c4 + 2] = fmaf(ri * __uint_as_float(raw[4 * c4 + 2]), c4v.z, s4.z);
            v[4 * c4 + 3] = fmaf(ri * __uint_as_float(raw[4 * c4 + 3]), c4v.w, s4.w);
          }
        }
        // segmented search: a chunk inside every window of the warp's rows costs one warp-uniform test; one that crosses a
        // window edge masks the columns outside each row's own window (they then never enter a set: +inf is the empty key)
        if constexpr (SEG) {
          if (!(j0 >= w_lo && j0 + TC_CHUNK <= w_hi)) {
#pragma unroll
            for (int c = 0; c < TC_CHUNK; ++c)
              if (j0 + c < my_lo || j0 + c >= my_hi) v[c] = INFINITY;
          }
        }
        if (diag && j0 < wrow0 + 32 && j0 + TC_CHUNK > wrow0) {  // warp-uniform, true for at most 2 chunks of one unit
#pragma unroll
          for (int c = 0; c < TC_CHUNK; ++c)
            if (j0 + c == gi) v[c] = INFINITY;  // self is slot 0 by construction (knn_finish)
        }
        if (fresh_set) {  // warp-uniform: the first 32 columns of a new row tile fill the 32 slots directly
          fresh_set = false;
          if (P.debug >= 1) return;
          uint32_t kv[TC_CHUNK];
#pragma unroll
          for (int c = 0; c < TC_CHUNK; ++c) {
            kv[c] = (__float_as_uint(v[c]) & ~31u) | (uint32_t)c;
            Lk[c * 32] = kv[c];
            Li[c * 32] = j0 + c;
          }
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const uint32_t a = max(max(kv[8 * t], kv[8 * t + 1]), max(kv[8 * t + 2], kv[8 * t + 3]));
            const uint32_t bq = max(max(kv[8 * t + 4], kv[8 * t + 5]), max(kv[8 * t + 6], kv[8 * t + 7]));
            gk[t] = max(a, bq);
          }
          smax = __uint_as_float(max(max(gk[0], gk[1]), max(gk[2], gk[3])) & ~31u);
          thr = fminf(smax, tlim);
          return;
        }
        // Steady state: no column of the chunk beats any row's threshold.  One min per element and one vote decide that; the
        // per-column hit mask (three instructions per element) is only built for chunks that do have a survivor.  On the
        // 1M-node graph the kernel runs under the power cap, where every SIMT instruction saved is tensor-pipe clock.
        float vm[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) vm[t] = fminf(fminf(v[4 * t], v[4 * t + 1]), fminf(v[4 * t + 2], v[4 * t + 3]));
        const float vmin = fminf(fminf(fminf(vm[0], vm[1]), fminf(vm[2], vm[3])), fminf(fminf(vm[4], vm[5]), fminf(vm[6], vm[7])));
        if (__any_sync(FULL, vmin < thr) && P.debug < 1) {
#pragma unroll
          for (int c = 0; c < TC_CHUNK; ++c) hits |= (v[c] < thr) ? (1u << c) : 0u;
        }
        // ---- every row (thread) inserts its own survivors; rows proceed concurrently ----
        while (__any_sync(FULL, hits != 0)) {
          ++nround;
          if (hits) {
            const int c = __ffs(hits) - 1;
            hits &= hits - 1;
            // The whole insertion is latency-bound (one warp's dependent chain), so every selection below is a balanced
            // tree, not a scan: v[c] by the bits of c (depth 5 instead of 31) ...
            float s16[16], s8[8], s4[4];
#pragma unroll
            for (int t = 0; t < 16; ++t) s16[t] = (c & 1) ? v[2 * t + 1] : v[2 * t];
#pragma unroll
            for (int t = 0; t < 8; ++t) s8[t] = (c & 2) ? s16[2 * t + 1] : s16[2 * t];
#pragma unroll
            for (int t = 0; t < 4; ++t) s4[t] = (c & 4) ? s8[2 * t + 1] : s8[2 * t];
            const float s2a = (c & 8) ? s4[1] : s4[0], s2b = (c & 8) ? s4[3] : s4[2];
            const float dsel = (c & 16) ? s2b : s2a;
            const uint32_t kbits = __float_as_uint(dsel) & ~31u;
            // second round (k > 33): the key is rebuilt exactly as the first round flushed it.  Admitted: every column whose
            // stored value is >= the first round's 32nd value, except that 32nd entry itself.  (Not "key > 32nd key": a column
            // that TIES with the 32nd value and has a smaller index may have been evicted from its set in the first round --
            // the entry a set drops among tied maxima is picked by slot, not by index -- and would be lost to both rounds.
            // First-round members that tie come back as duplicates; the re-rank drops them by index.)
            bool fresh = true;
            if (P.excl != nullptr) {
              const u64 key = make_key(unshift(__uint_as_float(kbits), sqi_row), j0 + c);
              fresh = (key != excl_row) && ((uint32_t)(key >> 32) >= (uint32_t)(excl_row >> 32));
            }
            if (dsel < thr && fresh) {  // thr may have tightened since the scan
              // replace the set's largest entry (one integer max over the four cached group maxima names it), reload its
              // group of eight and take the group's new maximum
              const uint32_t top = max(max(gk[0], gk[1]), max(gk[2], gk[3]));
              const int pos = (int)(top & 31u);
              Lk[pos * 32] = kbits | (uint32_t)pos;
              Li[pos * 32] = j0 + c;
              const uint32_t* grp = Lk + (pos & ~7) * 32;
              uint32_t tk[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) tk[e] = grp[e * 32];
              const uint32_t mx = max(max(max(tk[0], tk[1]), max(tk[2], tk[3])), max(max(tk[4], tk[5]), max(tk[6], tk[7])));
              const int g = pos >> 3;
#pragma unroll
              for (int t = 0; t < 4; ++t) gk[t] = (t == g) ? mx : gk[t];
              smax = __uint_as_float(max(max(gk[0], gk[1]), max(gk[2], gk[3])) & ~31u);
              thr = fminf(smax, tlim);
            }
          }
        }
      };
      // two register sets: the TMEM load of the next 32 columns is in flight while the current ones are processed
      constexpr int QH = TC_BN / TC_CHUNK / 2;  // chunks per warp (its half of the columns)
      static_assert(QH == 4, "the chunk loop below is written for four chunks per warp");
      const uint32_t tcol = taddr + (uint32_t)(half * (TC_BN / 2));
      auto hand_back = [&]() {  // this warp's half of the accumulator is in registers or consumed: the MMA warp may reuse it
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR)
            mbar_arrive_leader(bar_tempty + 8 * acc);  // the leader's MMA warp waits for both CTAs' epilogues
          else
            mbar_arrive(bar_tempty + 8 * acc);
        }
      };
      if (P.debug >= 2) {  // timing experiment: hand the accumulator back untouched
        hand_back();
      } else {
        tc_ld_issue(tcol, rawA);
        tc_ld_wait(rawA);
        tc_ld_issue(tcol + TC_CHUNK, rawB);
        process(rawA, 0);
        if (tg != 0xffffffffu) {
          // another set's bound, shifted (rounded up) and moved to the START OF THE NEXT five-bit bucket: a column whose
          // stored value would tie with that set's largest entry stays admissible.  (The completeness proof only needs the
          // statement on values -- every rejected column has a stored value >= the 32nd candidate's, tests/
          // test_candidate_sets_model.py -- which the plain bound gives as well; this keeps the merged list's tie order by
          // index intact wherever it can.)
          const float t_sh = __fadd_ru(ordered_to_float(tg + 1u), Cs);
          if (t_sh < INFINITY) {  // nothing published yet: +inf (or the NaN one past it)
            tlim = fminf(tlim, __uint_as_float((__float_as_uint(t_sh) | 31u) + 1u));
            thr = fminf(smax, tlim);
          }
        }
        tc_ld_wait(rawB);
        tc_ld_issue(tcol + 2 * TC_CHUNK, rawA);
        process(rawB, 1);
        tc_ld_wait(rawA);
        tc_ld_issue(tcol + 3 * TC_CHUNK, rawB);
        process(rawA, 2);
        tc_ld_wait(rawB);
        hand_back();
        process(rawB, 3);
      }
      if (tw > 0) {
        stamp(tw, u - u_begin, 4, clock64());
        stamp(tw, u - u_begin, 5, nround);
      }
      if (P.thr_g != nullptr && gi < P.n && smax < published) {  // my set is full and its bound improved during this unit
        atomicMin(P.thr_g + gi, float_to_ordered(__fadd_ru(smax, -Cs)));  // unshifted, rounded up: still an upper bound
        published = smax;
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1u;
    }
    if (cur_rt >= 0) flush(cur_rt);
  }

  tc_fence_before();
  if (PAIR)
    cluster_sync_all();  // nobody exits while the peer may still multicast into it or signal its barriers
  else
    __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TC_TMEM_COLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TC_TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- verification kernel
// ONE (row tile, column tile) unit with the production operand maps, descriptors and MMA sequence, but no pipeline and no
// epilogue: the raw fp32 accumulator goes to global memory so that a test can compare what the tensor core accumulated
// with the numpy model of the split (oracle/split_model.py) -- in particular that fp16 subnormal operands take part.
constexpr size_t TCD_OFF_BAR = TC_STAGE_BYTES;
constexpr size_t TCD_SMEM_BYTES = TCD_OFF_BAR + 64 + 1024;

__global__ void __launch_bounds__(128, 1)
knn_gram_tile_debug_kernel(const __grid_constant__ CUtensorMap mapAH, const __grid_constant__ CUtensorMap mapAL,
                           const __grid_constant__ CUtensorMap mapBH, int kblocks, int rt, int ct, int passes,
                           float* __restrict__ out) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t bar_full = base + (uint32_t)TCD_OFF_BAR, bar_mma = bar_full + 8, slot = bar_full + 16;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + TCD_OFF_BAR + 16);
  if (threadIdx.x == 0) {
    mbar_init(bar_full, 1);
    mbar_init(bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"((uint32_t)TC_BN) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t a_bytes = passes == 2 ? 2u * TC_A_BYTES : (uint32_t)TC_A_BYTES;
  const uint32_t stage_bytes = a_bytes + (uint32_t)TC_B_BYTES;
  const int nprod = passes;
  const uint32_t idesc = TC_IDESC_F16;
  uint32_t phase = 0;
  for (int kk = 0; kk < kblocks; ++kk) {
    if (threadIdx.x == 0) {
      mbar_arrive_expect_tx(bar_full, stage_bytes);
      tma_load_2d(base, &mapAH, bar_full, kk * TC_BK, rt * TC_BM);
      if (passes == 2) tma_load_2d(base + TC_A_BYTES, &mapAL, bar_full, kk * TC_BK, rt * TC_BM);
      tma_load_2d(base + a_bytes, &mapBH, bar_full, kk * TC_BK, ct * TC_BN);
    }
    mbar_wait(bar_full, phase);
    tc_fence_after();
    if (threadIdx.x == 0) {
      const uint64_t dAH = tc_smem_desc(base), dAL = tc_smem_desc(base + TC_A_BYTES);
      const uint64_t dBH = tc_smem_desc(base + a_bytes);
      for (int g = 0; g < nprod; ++g) {
        const uint64_t da = (g == 1) ? dAL : dAH, db = dBH;
        for (int k4 = 0; k4 < TC_BK / 16; ++k4)
          tc_mma_f16(tmem_base, da + (uint64_t)(2 * k4), db + (uint64_t)(2 * k4), idesc, (uint32_t)((kk | g | k4) != 0));
      }
      tc_commit(bar_mma);
    }
    mbar_wait(bar_mma, phase);  // the MMAs have retired: the stage may be overwritten, and after the last block D is complete
    tc_fence_after();
    phase ^= 1u;
  }
  const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
  uint32_t r[TC_CHUNK];
  for (int q = 0; q < TC_BN / TC_CHUNK; ++q) {
    tc_ld_issue(taddr + q * TC_CHUNK, r);
    tc_ld_wait(r);
#pragma unroll
    for (int c = 0; c < TC_CHUNK; ++c) out[(size_t)(warp * 32 + lane) * TC_BN + q * TC_CHUNK + c] = __uint_as_float(r[c]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TC_BN) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- host side
PFN_cuTensorMapEncodeTiled get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(p);
  }
  return fn;
}

int make_map(CUtensorMap* m, const void* base, int n, int d_pad, int box_rows) {
  PFN_cuTensorMapEncodeTiled enc = get_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from this driver");
    return GLL_ERR_CUDA;
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)d_pad, (cuuint64_t)n};
  const cuuint64_t gstride[1] = {(cuuint64_t)d_pad * 2};
  const cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, (TC_BK == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (n=%d d_pad=%d box_rows=%d)", (int)r, n, d_pad, box_rows);
    return GLL_ERR_CUDA;
  }
  return GLL_OK;
}

}  // namespace

TcPlan knn_tc_plan(int n, int d, int row_begin, int row_end, int col_begin) {
  TcPlan p;
  memset(&p, 0, sizeof(p));
  const char* force = getenv("GLL_B200_KNN_PATH");  // "simt" or "tc": testing knob, both paths are exact
  if (force && strcmp(force, "simt") == 0) return p;
  if (n < 2 * TC_BM && !(force && strcmp(force, "tc") == 0)) return p;  // tiny graphs: the SIMT kernel is enough
  if (row_begin % TC_BM != 0) return p;                                   // row ranges start on a tile boundary
  p.d_pad = ceil_div(d, TC_BK) * TC_BK;
  p.kblocks = p.d_pad / TC_BK;
  p.rt0 = row_begin / TC_BM;
  const int row_tiles = ceil_div(row_end - row_begin, TC_BM);
  const int sms = device_info().sms;
  p.ct0 = col_begin / TC_BN;
  p.col_begin = col_begin;
  p.col_tiles = ceil_div(n, TC_BN) - p.ct0;
  p.aligned = (row_tiles >= 4 * sms) ? 1 : 0;  // big graphs: whole row tiles per CTA, one candidate set per row
  // GLL_B200_KNN_PAIR: CTA pairs (clusters of 2, tcgen05.mma.cta_group::2 with M = 256): a third fewer operand bytes per CTA.
  const char* pr = getenv("GLL_B200_KNN_PAIR");
  // Default: from 64 row tiles (8192 rows) up -- measured -1 % at 10512 x 512, -6 % at 16384 x 512, -4 % at 32768 x 256, -10 % on
  // the 1M-node graph, no difference at 4608 x 512 (profiles/r02zm_knn_pair.txt)
  const bool pair = pr ? (pr[0] == '1') : (p.aligned != 0 || row_tiles >= 64);
  p.rstep = (pair && row_tiles >= 2 && sms >= 2) ? 2 : 1;
  p.row_tiles = ceil_div(row_tiles, p.rstep);  // row groups: the unit of work is (row group, column tile)
  p.units = (long long)p.row_tiles * p.col_tiles;
  const int owners = sms / p.rstep;
  p.grid = (int)((p.units < (long long)owners) ? p.units : (long long)owners);  // owners (CTAs or CTA pairs)
  // few row tiles (a batch-rows-only search): a row tile may be shared by at most KNN_MAX_SPLITS / 2 owners (two candidate
  // sets per owner and row), so the grid shrinks rather than the plan failing
  if (!p.aligned) p.grid = max(1, min(p.grid, p.row_tiles * (KNN_MAX_SPLITS / 2 - 1)));
  if (p.aligned) {
    p.max_splits = 2;  // the two column halves of the epilogue (knn_tc.cu: `half`)
  } else {
    int ms = 1;
    for (int rt = 0; rt < p.row_tiles; ++rt) {  // exact: owners touching each row group
      const int b0 = tc_cta_of_unit((long long)rt * p.col_tiles, p.grid, p.units);
      const int b1 = tc_cta_of_unit((long long)(rt + 1) * p.col_tiles - 1, p.grid, p.units);
      ms = max(ms, b1 - b0 + 1);
    }
    p.max_splits = 2 * ms;  // two candidate sets (column halves) per CTA and row
  }
  p.ws_bytes = 2 * align_up((size_t)n * p.d_pad * 2, 256);  // hi and (two passes) lo
  p.ok = (p.max_splits <= KNN_MAX_SPLITS) ? 1 : 0;
  // MMA passes over the fp16 operands: 1 = hi.hi (default), 2 = (hi + lo).hi (GLL_B200_KNN_SPLIT=f16x2).  Both only SELECT
  // candidates; the emitted lists are exact either way (the measured residual rho enters the completeness proof).
  const char* sp = getenv("GLL_B200_KNN_SPLIT");
  p.passes = (sp && strcmp(sp, "f16x2") == 0) ? 2 : 1;
  return p;
}

// Segmented unit grid: row group g (rstep row tiles) gets the column tiles that meet [lo of its first row, hi of its last row)
// -- segments are contiguous row ranges, so that is the union of its rows' windows.  Units are dealt to the owners exactly as
// in the uniform grid (contiguously, tc_cta_of_unit); the kernel, the flush slots and the re-rank all read gfirst.
TcPlan knn_tc_plan_segments(int n, int d, const int* seg_ptr, int nseg, std::vector<int>* tab) {
  TcPlan p = knn_tc_plan(n, d, 0, n);
  if (p.d_pad == 0) return p;  // SIMT path (tiny graph or forced)
  const int RG = p.row_tiles, rows_g = TC_BM * p.rstep;
  std::vector<int> gfirst(RG + 1), gct(RG);
  int s = 0, max_cnt = 1;
  long long units = 0;
  for (int g = 0; g < RG; ++g) {
    const int r0 = g * rows_g, r1 = std::min(n, r0 + rows_g) - 1;
    while (seg_ptr[s + 1] <= r0) ++s;
    const int lo = seg_ptr[s];
    int t = s;
    while (seg_ptr[t + 1] <= r1) ++t;
    const int hi = seg_ptr[t + 1];
    gct[g] = lo / TC_BN;
    const int cnt = ceil_div(hi, TC_BN) - gct[g];
    gfirst[g] = (int)units;
    units += cnt;
    max_cnt = std::max(max_cnt, cnt);
  }
  gfirst[RG] = (int)units;
  (void)nseg;
  p.units = units;
  p.col_tiles = max_cnt;
  const int owners = device_info().sms / p.rstep;
  p.grid = (int)std::min<long long>(units, owners);
  std::vector<int> bstart;
  for (;;) {
    if (!p.aligned) p.grid = std::max(1, std::min(p.grid, RG * (KNN_MAX_SPLITS / 2 - 1)));
    int ms = 1;
    if (!p.aligned)
      for (int g = 0; g < RG; ++g)
        ms = std::max(ms, tc_cta_of_unit(gfirst[g + 1] - 1, p.grid, units) - tc_cta_of_unit(gfirst[g], p.grid, units) + 1);
    p.max_splits = 2 * ms;
    if (p.max_splits <= KNN_MAX_SPLITS || p.grid == 1) break;
    p.grid = std::max(1, p.grid * 3 / 4);  // a long row group shared by too many owners: fewer owners
  }
  p.ok = (p.max_splits <= KNN_MAX_SPLITS) ? 1 : 0;
  bstart.resize(p.grid);
  for (int b = 0, g = 0; b < p.grid; ++b) {
    const long long u0 = (long long)b * units / p.grid;
    while (g + 1 < RG && gfirst[g + 1] <= u0) ++g;
    bstart[b] = g;
  }
  tab->clear();
  tab->insert(tab->end(), gfirst.begin(), gfirst.end());
  tab->insert(tab->end(), gct.begin(), gct.end());
  tab->insert(tab->end(), bstart.begin(), bstart.end());
  return p;
}

size_t knn_tc_ws_upper(int n, int d) { return 2 * align_up((size_t)n * (size_t)(ceil_div(d, TC_BK) * TC_BK) * 2, 256) + 512; }

// |d~^2 - d^2| <= coef (|xi|^2 + max|x|^2) + [the rho term of knn_err_bound()].  coef budgets what rho does not measure:
//  * fp16 SUBNORMAL operand elements, in case the multiplier flushed them: rows are scaled to a norm of at least 148, so an
//    element below fp16's normal range is below 2^-14 2^E_i <= 2^-21.2 |x_i|; over d elements that is at most
//    2^-21.2 sqrt(d) |x_i| per operand whose rounding is not already in rho (two passes: the A side, whose hi + lo is exact
//    to 2^-22 |x_ik| elsewhere; one pass: budgeted for both sides, although rho measures hi's own rounding exactly);
//  * fp32 accumulation over passes * d/16 MMA steps of unknown internal rounding (2^-21 per step and per 16-term tree);
//  * the final fp32 expression, 4u;  then a 4x margin.
float knn_tc_err_coef(int d, int passes) {
  const double steps = (double)passes * ceil_div(d, 16) + 8.0;
  const double split = (passes == 1 ? 2.0 : 1.0) * (1.0 + sqrt((double)d)) / 2097152.0 * 1.01;
  // 12 ulps: the roundings of the epilogue (|x_j|^2 + Cs, the FMA at the magnitude of the shifted value, un-shifting and
  // adding |x_i|^2 when a set is flushed: <= 15 * 2^-24 max|x|^2 together, against 4 * 12 * 2^-24 (|x_i|^2 + max|x|^2) here)
  const double e = split + steps * 4.76837158203125e-7 + 12.0 * 5.9604644775390625e-8;
  return (float)(4.0 * e);
}

int knn_tc_debug_tile(const TcPlan& plan, int n, void* tc_ws, int rt, int ct, float* acc_out, cudaStream_t st) {
  __half* H = reinterpret_cast<__half*>(tc_ws);
  __half* L = reinterpret_cast<__half*>((char*)tc_ws + align_up((size_t)n * plan.d_pad * 2, 256));
  CUtensorMap mAH, mAL, mBH;
  int rc;
  if ((rc = make_map(&mAH, H, n, plan.d_pad, TC_BM))) return rc;
  if ((rc = make_map(&mAL, L, n, plan.d_pad, TC_BM))) return rc;
  if ((rc = make_map(&mBH, H, n, plan.d_pad, TC_BN))) return rc;
  GLL_CUDA_CHECK(set_max_dynamic_smem_once((const void*)knn_gram_tile_debug_kernel, (int)TCD_SMEM_BYTES));
  knn_gram_tile_debug_kernel<<<1, 128, TCD_SMEM_BYTES, st>>>(mAH, mAL, mBH, plan.kblocks, rt, ct, plan.passes, acc_out);
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

static unsigned long long* g_knn_trace = nullptr;  // debug only: [TC_TRACE_WARPS][TC_TRACE_UNITS][TC_TRACE_PHASES] of CTA 0
void knn_tc_set_trace(void* device_buf) { g_knn_trace = reinterpret_cast<unsigned long long*>(device_buf); }

int knn_tc_candidates(const float* X, const float* sq, const float* rscale, const unsigned* small, int n, int d, int row_end, const TcPlan& plan,
                      void* tc_ws, u64* cand, const u64* excl, unsigned* thr_g, cudaStream_t st, const SegDev* seg) {
  __half* H = reinterpret_cast<__half*>(tc_ws);
  __half* L = reinterpret_cast<__half*>((char*)tc_ws + align_up((size_t)n * plan.d_pad * 2, 256));
  // H and L (fp16 hi / lo of the scaled rows, row stride d_pad) were written by sqnorm_split_f16_kernel (knn.cu); with one
  // pass L is never touched (the map is encoded over the same allocation)
  CUtensorMap mAH, mAL, mBH;
  int rc;
  if ((rc = make_map(&mAH, H, n, plan.d_pad, TC_BM))) return rc;
  if ((rc = make_map(&mAL, L, n, plan.d_pad, TC_BM))) return rc;
  if ((rc = make_map(&mBH, H, n, plan.d_pad, TC_BN))) return rc;
  TcParams P;
  P.n = n;
  P.kblocks = plan.kblocks;
  P.col_tiles = plan.col_tiles;
  P.max_splits = plan.max_splits;
  P.units = plan.units;
  P.rt0 = plan.rt0;
  P.row_end = row_end;
  P.ct0 = plan.ct0;
  P.col_begin = plan.col_begin;
  P.aligned = plan.aligned;
  P.row_tiles = plan.row_tiles;
  P.sq = sq;
  P.cand = cand;
  P.excl = excl;
  P.thr_g = thr_g;
  P.passes = plan.passes;
  P.rscale = rscale;
  P.small = small;
  const bool segd = seg != nullptr;
  SegDev S;
  if (segd) S = *seg;
  else memset(&S, 0, sizeof(S));
  {
    const char* dbg = getenv("GLL_B200_KNN_DEBUG");
    P.debug = dbg ? atoi(dbg) : 0;
  }
  P.trace = g_knn_trace;
  {
    // resident A operand: when all K blocks of a row tile and at least three B stages fit the stage region (d <= 384 with CTA
    // pairs and one pass); default in the large-graph mode (a row tile is swept over all column tiles), GLL_B200_KNN_ARES=0/1
    const size_t need = (size_t)plan.kblocks * a_bytes_of(plan.passes) + 3u * (size_t)(plan.rstep == 2 ? TC_B_BYTES / 2 : TC_B_BYTES);
    const bool fits = need <= TC_STAGE_REGION;
    const char* e = getenv("GLL_B200_KNN_ARES");
    P.ares = (fits && (e ? atoi(e) != 0 : plan.aligned != 0)) ? 1 : 0;
  }
  auto kern = segd ? (plan.rstep == 2 ? knn_gram_topk_tc_kernel<true, true> : knn_gram_topk_tc_kernel<false, true>)
                   : (plan.rstep == 2 ? knn_gram_topk_tc_kernel<true, false> : knn_gram_topk_tc_kernel<false, false>);
  GLL_CUDA_CHECK(set_max_dynamic_smem_once((const void*)kern, (int)TC_SMEM_BYTES));
  {
    GLL_PROF(KID_GRAM_TOPK_TC, st);
    if (plan.rstep == 2) {
      cudaLaunchConfig_t cfg;
      memset(&cfg, 0, sizeof(cfg));
      cfg.gridDim = dim3(2 * plan.grid);
      cfg.blockDim = dim3(TC_THREADS);
      cfg.dynamicSmemBytes = TC_SMEM_BYTES;
      cfg.stream = st;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2;
      attr[0].val.clusterDim.y = 1;
      attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      GLL_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, mAH, mAL, mBH, P, S));
    } else {
      kern<<<plan.grid, TC_THREADS, TC_SMEM_BYTES, st>>>(mAH, mAL, mBH, P, S);
    }
  }
  GLL_LAUNCH_CHECK();
  return GLL_OK;
}

}  // namespace gll
