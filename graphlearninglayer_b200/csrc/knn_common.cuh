// Pieces shared by the SIMT (knn.cu) and tensor-core (knn_tc.cu) kNN candidate kernels.
#pragma once
#include <vector>

#include "common.cuh"

namespace gll {

typedef unsigned long long u64;
constexpr int KC = 32;               // candidates kept per row (one per lane)
constexpr int KNN_MAX_SPLITS = 32;   // candidate lists per row: two per CTA that touches the row tile
constexpr u64 KEY_INF = ~0ull;

// key = (order-preserving bits of the approximate squared distance, column index): u64 compare == (dist, idx) compare
__device__ __forceinline__ u64 make_key(float dist, int j) {
  return ((u64)float_to_ordered(dist) << 32) | (uint32_t)j;
}
__device__ __forceinline__ float key_dist(u64 k) { return ordered_to_float((uint32_t)(k >> 32)); }
__device__ __forceinline__ int key_idx(u64 k) { return (int)(uint32_t)k; }

// Insert x into an ascending list of 32 keys held one per lane (keys are unique). No-op if x is larger than all.
__device__ __forceinline__ void list_insert(u64& mine, u64 x, int lane) {
  int pos = __popc(__ballot_sync(FULL, mine < x));
  u64 prev = __shfl_up_sync(FULL, mine, 1);
  if (lane > pos)
    mine = prev;
  else if (lane == pos)
    mine = x;
}

// compare-exchange with the lane at xor distance j: keep the smaller key if keep_min
__device__ __forceinline__ void key_cmpx(u64& k, int j, bool keep_min) {
  const u64 o = __shfl_xor_sync(FULL, k, j);
  const bool less = k < o;
  k = (less == keep_min) ? k : o;
}
// ascending bitonic sort of 32 keys, one per lane
__device__ __forceinline__ void key_sort32(u64& k, int lane) {
#pragma unroll
  for (int w = 2; w <= 32; w <<= 1) {
#pragma unroll
    for (int j = w >> 1; j >= 1; j >>= 1) {
      const bool up = (lane & w) == 0;  // w == 32: every lane ascending
      key_cmpx(k, j, ((lane & j) == 0) == up);
    }
  }
}
// Merge one unsorted 32-set (one key per lane, KEY_INF = empty) into the sorted list `mine`.  Only keys below the list's
// current last entry can enter: a handful are inserted one by one (one ballot finds them); many -- the first lists of a
// row -- go through a sorting network: sort the set, take min(mine[i], set[31 - i]) (the 32 smallest of the union, a
// bitonic sequence) and merge it back into ascending order.  The serial form alone was 40 % of the re-rank kernel's
// instructions.
__device__ __forceinline__ void list_merge_set(u64& mine, u64 c, int lane) {
  unsigned m = __ballot_sync(FULL, c < __shfl_sync(FULL, mine, KC - 1));
  if (m == 0) return;
  if (__popc(m) > 6) {
    key_sort32(c, lane);
    const u64 r = __shfl_sync(FULL, c, 31 - lane);
    mine = (r < mine) ? r : mine;
#pragma unroll
    for (int j = 16; j >= 1; j >>= 1) key_cmpx(mine, j, (lane & j) == 0);
    return;
  }
  while (m) {
    const int t = __ffs(m) - 1;
    m &= m - 1;
    const u64 x = __shfl_sync(FULL, c, t);
    if (x < __shfl_sync(FULL, mine, KC - 1)) list_insert(mine, x, lane);  // the last entry may have tightened meanwhile
  }
}

// Tensor-core candidate generation (knn_tc.cu).  plan.ok == 0: shape or configuration not handled, use the SIMT path.
struct TcPlan {
  int ok, d_pad, kblocks, row_tiles, col_tiles, grid, max_splits, rt0, aligned, rstep;  // row_tiles counts row GROUPS of rstep tiles
  int ct0, col_begin;  // column range [col_begin, n): first column tile; columns before col_begin inside it are masked
  int passes;       // MMA passes over the fp16 operands (rows of X scaled by a power of two): 1 = hi.hi, 2 = (hi + lo).hi
  long long units;
  size_t ws_bytes;  // fp16 hi / lo copies of X
};

// Segmented search (gll_knn_segments): row i only sees the columns of its own segment, win[i] = [lo, hi).  The tensor-core
// unit grid then has, per row group g, only the column tiles [gct[g], gct[g] + gfirst[g + 1] - gfirst[g]) that meet the
// windows of its rows; units are numbered row group by row group (gfirst[g] = first unit of g), and bstart[b] is the row
// group of owner b's first unit.  Device arrays in the workspace; all NULL for an unsegmented search.
struct SegDev {
  const int2* win;
  const int* gfirst;
  const int* gct;
  const int* bstart;
};

TcPlan knn_tc_plan(int n, int d, int row_begin, int row_end, int col_begin = 0);
// the plan of a segmented search over all n rows; *tab receives gfirst, gct and bstart (in that order, see SegDev)
TcPlan knn_tc_plan_segments(int n, int d, const int* seg_ptr, int nseg, std::vector<int>* tab);
size_t knn_tc_ws_upper(int n, int d);
int knn_tc_candidates(const float* X, const float* sq, const float* rscale, const unsigned* small, int n, int d, int row_end, const TcPlan& plan,
                      void* tc_ws, u64* cand, const u64* excl, unsigned* thr_g, cudaStream_t st, const SegDev* seg = nullptr);
float knn_tc_err_coef(int d, int passes);
// verification: raw accumulator of one (row tile, column tile) unit, acc_out[128][256] (knn_gram_tile_debug_kernel)
int knn_tc_debug_tile(const TcPlan& plan, int n, void* tc_ws, int rt, int ct, float* acc_out, cudaStream_t st);

// How the candidate lists of a row are laid out in cand[n][stride][KC]: uniform (SIMT: every row has `stride` lists)
// or the tensor-core work split (row tile rt was touched by CTAs b0(rt)..b1(rt); slot = b - b0).
struct CandLayout {
  int stride;      // lists allocated per row
  int tc;          // 0: every row has `stride` sorted lists; 1: tensor-core work split; 2: one unsorted set per row;
                   // 3: tensor-core work split over a segmented unit grid (row group g owns units [gfirst[g], gfirst[g + 1]))
  int row_begin;   // first row of this call's row range (row tiles are counted from it)
  int row_tile, col_tiles, grid;
  long long units;
  const int* gfirst;  // tc == 3 only (SegDev::gfirst)
};

// CTAs of a G-CTA tensor-core launch over `units` units that wrote candidate sets for row group rt: b0 .. b1
__device__ __forceinline__ void cand_owner_range(const CandLayout& lay, long long rt, int& b0, int& b1) {
  const long long f0 = (lay.tc == 3) ? (long long)__ldg(lay.gfirst + rt) : rt * lay.col_tiles;
  const long long f1 = (lay.tc == 3) ? (long long)__ldg(lay.gfirst + rt + 1) : (rt + 1) * lay.col_tiles;
  b0 = (int)(((f0 + 1) * lay.grid - 1) / lay.units);
  b1 = (int)((f1 * lay.grid - 1) / lay.units);
}

// candidate lists written for row i: `stride`, or under the tensor-core work split two per CTA that touched the row's group
// (the column halves of its epilogue)
__device__ __forceinline__ int cand_lists(const CandLayout& lay, int i) {
  if (lay.tc != 1 && lay.tc != 3) return lay.stride;
  int b0, b1;
  cand_owner_range(lay, (i - lay.row_begin) / lay.row_tile, b0, b1);
  return 2 * (b1 - b0 + 1);
}

}  // namespace gll
