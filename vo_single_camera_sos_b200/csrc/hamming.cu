// Step 2 of the SOS front-end: brute-force Hamming matching of 256-bit ORB descriptors.
//
// Replaces cv2.BFMatcher(NORM_HAMMING).match / knnMatch(k=2) as used by FeatureMatcher.match
// (reference omnistereo/camera_models.py:402-446), the post-sort at camera_models.py:444 and the pixel gate
// filter_pixel_correspondences (common_cv.py:167-188).
//
// Kernel design (integer-pipe bound, SURVEY §8d):
//   * a thread keeps QPT query descriptors in registers (8 x u32 each);
//   * the block stages a tile of train descriptors in shared memory; every lane reads the SAME train
//     descriptor (two broadcast LDS.128), so shared-memory traffic is 32 B per 32*QPT descriptor pairs;
//   * per pair: 8 LOP3(xor) + 8 POPC + 4 IADD3, then a branch-free top-2 update on the packed key
//     (distance << 22 | train index) — min/max on the key gives OpenCV's (distance, lowest index) order;
//   * the train range of a segment is split over blockIdx.y so that small problems still fill 148 SMs;
//     the per-split partial keys are merged by a second, tiny kernel.
#include <stdlib.h>

#include "sos_common.cuh"

// tensor-core engine (hamming_mma.cu)
size_t sos_hamming_mma_scratch_bytes(int n_seg, int max_nq, int max_nt);
int sos_hamming_mma_launch(sos_ctx* ctx, const uint32_t* q, const uint32_t* t, const int32_t* q_start, const int32_t* q_len,
                           const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq, int max_nt, int splits,
                           const uint32_t* items, const int32_t* n_items, unsigned max_items, bool top2, void* exp,
                           uint2* partial);

size_t sos_l2_mma_scratch_bytes(int n_seg, int max_nq, int max_nt);
int sos_l2_mma_launch(sos_ctx* ctx, const float* q, const float* t, int dim, const int32_t* q_start, const int32_t* q_len,
                      const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq, int max_nt, int splits,
                      const uint32_t* items, const int32_t* n_items, unsigned max_items, bool top2, void* exp,
                      ulonglong2* partial, int32_t* flag);

size_t sos_l2f_scratch_bytes(int n_seg, int max_nq, int max_nt, int dim, int splits);
int sos_l2f_launch(sos_ctx* ctx, const float* q, const float* t, int dim, const int32_t* q_start, const int32_t* q_len,
                   const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq, int max_nt, int splits,
                   const uint32_t* items, const int32_t* n_items, unsigned max_items, bool top2, void* scratch,
                   int32_t* idx0, float* d0, int32_t* idx1, float* d1, int32_t* flag, int32_t* stats);

namespace {

constexpr int HB_THREADS = 128;  // threads per block
constexpr int HB_QPT = 2;        // query descriptors per thread
constexpr int HB_TILE_Q = HB_THREADS * HB_QPT;
constexpr int HB_TILE_T = 256;   // train descriptors per shared-memory tile (8 KB)
constexpr int KEY_IDX_BITS = 22; // up to 4M train rows per segment; distance <= 256 needs 9 bits
constexpr uint32_t KEY_NONE = 0xFFFFFFFFu;

// carry-save adder on 32 bit lanes: a + b + c = sum + 2 * carry (one LOP3 each)
// Written as two explicit LOP3s (truth tables 0x96 = a^b^c, 0xE8 = majority): left to itself the compiler re-factors
// the boolean network together with the XORs feeding it and ends up with ~50 % more LOP3s (measured in SASS), which
// makes the ALU pipe the bottleneck instead of the XU pipe.
__device__ __forceinline__ void csa(uint32_t a, uint32_t b, uint32_t c, uint32_t& sum, uint32_t& carry) {
  asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(sum) : "r"(a), "r"(b), "r"(c));
  asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(carry) : "r"(a), "r"(b), "r"(c));
}

// Packed key (distance << KEY_IDX_BITS) + tj of one descriptor pair.  Three carry-save adders first, then 5 POPC instead
// of 8: moves work from the XU pipe (POPC, 16 lanes/clk/SM: the narrow pipe) to the 4x wider ALU pipe; the weighted sum
// and the key are formed by IMADs on the FMA pipe.  (Measured against plain 8 x POPC and a full Harley-Seal tree with
// 4 POPC in round 1: this one is the fastest, profiles/r01/.)
__device__ __forceinline__ uint32_t hamming_key(const uint4& qa, const uint4& qb, const uint4& ta, const uint4& tb,
                                                uint32_t tj) {
  const uint32_t x0 = qa.x ^ ta.x, x1 = qa.y ^ ta.y, x2 = qa.z ^ ta.z, x3 = qa.w ^ ta.w;
  const uint32_t x4 = qb.x ^ tb.x, x5 = qb.y ^ tb.y, x6 = qb.z ^ tb.z, x7 = qb.w ^ tb.w;
  uint32_t s1, c1, s2, c2, s3, c3;
  csa(x0, x1, x2, s1, c1);
  csa(x3, x4, x5, s2, c2);
  csa(s1, s2, x6, s3, c3);
  const uint32_t ones = __popc(s3) + __popc(x7);
  const uint32_t twos = __popc(c1) + __popc(c2) + __popc(c3);
  return twos * (2u << KEY_IDX_BITS) + (ones * (1u << KEY_IDX_BITS) + tj);
}

// Work list: segment lengths live on the device, so the host can only size the grid for the worst case.  Launching
// that grid directly leaves the SMs unevenly loaded (blocks of short segments exit at once and everything fits in
// one wave: measured 66 % average SM activity).  Instead one small block compacts the ACTIVE (segment, query tile,
// train split) items into a list; block i of the main kernel takes item i, so the active blocks are contiguous in
// launch order and the hardware scheduler balances them.
constexpr int ITEM_SPLIT_BITS = 6, ITEM_TILE_BITS = 10;  // item = seg << 16 | tile << 6 | split

__global__ void __launch_bounds__(256)
hamming_plan_kernel(const int32_t* __restrict__ q_len, int n_seg, int max_nq, int splits, uint32_t* __restrict__ items,
                    int32_t* __restrict__ n_items) {
  __shared__ int warp_tot[8];
  __shared__ int carry_sh;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry_sh = 0;
  __syncthreads();
  for (int base = 0; base < n_seg; base += 256) {
    const int seg = base + tid;
    const int tiles = seg < n_seg ? (min(q_len[seg], max_nq) + HB_TILE_Q - 1) / HB_TILE_Q : 0;
    const int cnt = tiles * splits;
    int incl = cnt;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int v = __shfl_up_sync(0xFFFFFFFFu, incl, off);
      if (lane >= off) incl += v;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    int before = carry_sh;
    for (int w = 0; w < warp; ++w) before += warp_tot[w];
    const int first = before + incl - cnt;
    for (int k = 0; k < cnt; ++k)
      items[first + k] = ((uint32_t)seg << 16) | ((uint32_t)(k / splits) << ITEM_SPLIT_BITS) | (uint32_t)(k % splits);
    __syncthreads();
    if (tid == 255) carry_sh = before + incl;
    __syncthreads();
  }
  if (tid == 0) *n_items = carry_sh;
}

template <bool TOP2>
__global__ void __launch_bounds__(HB_THREADS)
hamming_partial_kernel(const uint4* __restrict__ q, const uint4* __restrict__ t, const int32_t* __restrict__ q_start,
                       const int32_t* __restrict__ q_len, const int32_t* __restrict__ t_start,
                       const int32_t* __restrict__ t_len, int max_nq, int max_nt, int splits,
                       const uint32_t* __restrict__ items, const int32_t* __restrict__ n_items, uint2* __restrict__ partial) {
  __shared__ uint4 tile[HB_TILE_T * 2];

  if ((int)blockIdx.x >= *n_items) return;
  const uint32_t item = items[blockIdx.x];
  const int seg = (int)(item >> 16);
  const int q0 = q_start[seg], nq = min(q_len[seg], max_nq);
  const int q_tile = (int)((item >> ITEM_SPLIT_BITS) & ((1u << ITEM_TILE_BITS) - 1u)) * HB_TILE_Q;
  const int t0 = t_start[seg], nt = min(t_len[seg], max_nt);
  const int split = (int)(item & ((1u << ITEM_SPLIT_BITS) - 1u));
  const int chunk = (nt + splits - 1) / splits;
  const int t_begin = min(nt, split * chunk);
  const int t_end = min(nt, t_begin + chunk);

  uint4 qa[HB_QPT], qb[HB_QPT];
  uint32_t k0[HB_QPT], k1[HB_QPT];
#pragma unroll
  for (int r = 0; r < HB_QPT; ++r) {
    int row = q_tile + r * HB_THREADS + threadIdx.x;
    if (row >= nq) row = nq - 1;  // clamp: computes a duplicate that is never stored
    const uint4* p = q + (size_t)(q0 + row) * 2;
    qa[r] = __ldg(p);
    qb[r] = __ldg(p + 1);
    k0[r] = KEY_NONE;
    k1[r] = KEY_NONE;
  }

  for (int tb = t_begin; tb < t_end; tb += HB_TILE_T) {
    const int n_tile = min(HB_TILE_T, t_end - tb);
    __syncthreads();
    const uint4* src = t + (size_t)(t0 + tb) * 2;
    for (int i = threadIdx.x; i < n_tile * 2; i += HB_THREADS) tile[i] = __ldg(src + i);
    __syncthreads();

    int j = 0;
    for (; j + 4 <= n_tile; j += 4) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint4 ta = tile[(j + u) * 2], tbv = tile[(j + u) * 2 + 1];
        const uint32_t tj = (uint32_t)(tb + j + u);
#pragma unroll
        for (int r = 0; r < HB_QPT; ++r) {
          const uint32_t key = hamming_key(qa[r], qb[r], ta, tbv, tj);
          if (TOP2) k1[r] = min(k1[r], max(k0[r], key));
          k0[r] = min(k0[r], key);
        }
      }
    }
    for (; j < n_tile; ++j) {
      const uint4 ta = tile[j * 2], tbv = tile[j * 2 + 1];
      const uint32_t tj = (uint32_t)(tb + j);
#pragma unroll
      for (int r = 0; r < HB_QPT; ++r) {
        const uint32_t key = hamming_key(qa[r], qb[r], ta, tbv, tj);
        if (TOP2) k1[r] = min(k1[r], max(k0[r], key));
        k0[r] = min(k0[r], key);
      }
    }
  }

#pragma unroll
  for (int r = 0; r < HB_QPT; ++r) {
    const int row = q_tile + r * HB_THREADS + threadIdx.x;
    if (row < nq) partial[((size_t)seg * max_nq + row) * splits + split] = make_uint2(k0[r], k1[r]);
  }
}

__global__ void __launch_bounds__(256)
hamming_merge_kernel(const uint2* __restrict__ partial, const int32_t* __restrict__ q_start,
                     const int32_t* __restrict__ q_len, int max_nq, int splits, int32_t* __restrict__ idx0,
                     int32_t* __restrict__ d0, int32_t* __restrict__ idx1, int32_t* __restrict__ d1) {
  const int seg = blockIdx.y;
  const int q0 = q_start[seg], nq = min(q_len[seg], max_nq);
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= nq) return;
  const uint2* p = partial + ((size_t)seg * max_nq + row) * splits;
  uint32_t k0 = KEY_NONE, k1 = KEY_NONE;
  for (int s = 0; s < splits; ++s) {
    const uint2 v = p[s];
    // merge two sorted pairs: v.x <= v.y
    k1 = min(k1, max(k0, v.x));
    k0 = min(k0, v.x);
    k1 = min(k1, v.y);  // v.y >= v.x, so it can only compete for second place
  }
  const uint32_t mask = (1u << KEY_IDX_BITS) - 1u;
  idx0[q0 + row] = (k0 == KEY_NONE) ? -1 : (int32_t)(k0 & mask);
  d0[q0 + row] = (k0 == KEY_NONE) ? -1 : (int32_t)(k0 >> KEY_IDX_BITS);
  if (idx1) idx1[q0 + row] = (k1 == KEY_NONE) ? -1 : (int32_t)(k1 & mask);
  if (d1) d1[q0 + row] = (k1 == KEY_NONE) ? -1 : (int32_t)(k1 >> KEY_IDX_BITS);
}

// ---------------------------------------------------------------------------------------------------
// match_select: mode filter + pixel gate + stable counting sort by (distance, query index).
// One block per segment.
// ---------------------------------------------------------------------------------------------------
constexpr int MS_THREADS = 1024;
constexpr int MS_WARPS = MS_THREADS / 32;
constexpr int MS_BINS = 257;

struct SelectArgs {
  int mode;
  double ratio;
  const int32_t *idx0, *d0, *d1, *rev_idx0, *q_start, *q_len, *t_start;
  const float2 *px_q, *px_t;
  double max_du, min_dv;
  int32_t *out_q, *out_t, *out_d, *out_count;
};

__device__ __forceinline__ bool select_keep(const SelectArgs& a, int q0, int t0, int q, int& t_local, int& dist) {
  t_local = a.idx0[q0 + q];
  dist = a.d0[q0 + q];
  if (t_local < 0) return false;
  if (a.mode == SOS_MATCH_RATIO) {
    const int dd1 = a.d1[q0 + q];
    if (dd1 < 0) return false;                                  // len(m) == 2 fails (camera_models.py:423)
    if (!((double)dist < (double)dd1 * a.ratio)) return false;
  } else if (a.mode == SOS_MATCH_CROSS) {
    if (a.rev_idx0[t0 + t_local] != q) return false;
  }
  if (a.px_q != nullptr) {
    const float2 pq = a.px_q[q0 + q];
    const float2 pt = a.px_t[t0 + t_local];
    if (a.max_du > 0.0 && !(fabs((double)pt.x - (double)pq.x) <= a.max_du)) return false;  // common_cv.py:177-178
    if (a.min_dv >= 0.0 && !((double)pt.y - (double)pq.y >= a.min_dv)) return false;       // common_cv.py:182-184
  }
  return true;
}

__global__ void __launch_bounds__(MS_THREADS) match_select_kernel(SelectArgs a) {
  __shared__ int hist[MS_BINS + 1];
  __shared__ int cursor[MS_BINS];
  __shared__ unsigned char warpcnt[MS_WARPS][MS_BINS + 3];

  const int seg = blockIdx.x;
  const int q0 = a.q_start[seg], nq = a.q_len[seg];
  const int t0 = a.t_start[seg];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  for (int i = tid; i <= MS_BINS; i += MS_THREADS) hist[i] = 0;
  for (int i = tid; i < MS_WARPS * (MS_BINS + 3); i += MS_THREADS) (&warpcnt[0][0])[i] = 0;
  __syncthreads();

  for (int q = tid; q < nq; q += MS_THREADS) {
    int tl, d;
    if (select_keep(a, q0, t0, q, tl, d)) atomicAdd(&hist[d], 1);
  }
  __syncthreads();
  // exclusive scan of 257 bins by one warp (9 bins per lane)
  if (warp == 0) {
    int local[9];
    int sum = 0;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const int b = lane * 9 + k;
      local[k] = (b < MS_BINS) ? hist[b] : 0;
      sum += local[k];
    }
    int incl = sum;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int v = __shfl_up_sync(0xFFFFFFFFu, incl, off);
      if (lane >= off) incl += v;
    }
    int run = incl - sum;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const int b = lane * 9 + k;
      if (b < MS_BINS) cursor[b] = run;
      run += local[k];
    }
    if (lane == 31) a.out_count[seg] = incl;
  }
  __syncthreads();

  const int n_chunks = (nq + MS_THREADS - 1) / MS_THREADS;
  for (int c = 0; c < n_chunks; ++c) {
    const int q = c * MS_THREADS + tid;
    int tl = -1, d = 0;
    const bool keep = (q < nq) && select_keep(a, q0, t0, q, tl, d);
    // rank among lanes of this warp with the same distance
    const unsigned vote = __ballot_sync(0xFFFFFFFFu, keep);
    unsigned same = 0;
    if (keep) same = __match_any_sync(vote, d);
    const int rank_in_warp = __popc(same & ((1u << lane) - 1u));
    const bool leader = keep && rank_in_warp == 0;
    if (leader) warpcnt[warp][d] = (unsigned char)__popc(same);
    __syncthreads();
    if (keep) {
      int before = 0;
      for (int w = 0; w < warp; ++w) before += warpcnt[w][d];
      const int pos = cursor[d] + before + rank_in_warp;
      a.out_q[q0 + pos] = q0 + q;
      a.out_t[q0 + pos] = t0 + tl;
      a.out_d[q0 + pos] = d;
    }
    __syncthreads();
    if (leader) {
      atomicAdd(&cursor[d], (int)warpcnt[warp][d]);
      warpcnt[warp][d] = 0;
    }
    __syncthreads();
  }
}

}  // namespace

extern "C" int sos_hamming_top2(sos_ctx* ctx, const uint32_t* q, const uint32_t* t, const int32_t* q_start,
                                const int32_t* q_len, const int32_t* t_start, const int32_t* t_len, int n_seg,
                                int max_nq, int max_nt, int32_t* idx0, int32_t* d0, int32_t* idx1, int32_t* d1) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n_seg >= 0 && max_nq >= 0 && max_nt >= 0, "negative size");
  SOS_CHECK_ARG(n_seg <= 65535, "at most 65535 segments per call");
  SOS_CHECK_ARG(max_nt < (1 << KEY_IDX_BITS), "segment has too many train rows (limit 4194303)");
  if (n_seg == 0 || max_nq == 0) return SOS_OK;
  SOS_CHECK_ARG(q && t && q_start && q_len && t_start && t_len && idx0 && d0, "NULL array");
  SOS_CHECK_ARG(((uintptr_t)q & 15) == 0 && ((uintptr_t)t & 15) == 0, "descriptor arrays must be 16-byte aligned");
  SOS_CUDA(cudaSetDevice(ctx->device));

  const int q_tiles = sos_div_up(max_nq, HB_TILE_Q);
  SOS_CHECK_ARG(q_tiles <= (1 << ITEM_TILE_BITS), "segment has too many query rows (limit 262144)");
  const bool top2 = idx1 != nullptr || d1 != nullptr;
  // engine: "popc" = XOR + POPC on the integer pipe, "mma" = int8 tensor cores (hamming_mma.cu).  Default: the tensor-core
  // engine once a segment can fill a few 128 x 128 tiles; below that its fixed cost (expansion, 180 KB of shared memory per
  // CTA, TMEM allocation) is not repaid.  SOS_HAMMING_ENGINE overrides (read per call; both engines run the same tests).
  const char* eng = getenv("SOS_HAMMING_ENGINE");
  bool use_mma = max_nq >= 256 && max_nt >= 512;
  if (eng && eng[0] == 'p') use_mma = false;
  if (eng && eng[0] == 'm') use_mma = max_nt > 0;

  int splits;
  if (use_mma) {
    // a work item is 256 query rows x (train tiles / splits); keep >= 4 train tiles per item (the two query tiles of an
    // item are fetched once per item) unless that starves the SMs
    const int t_tiles = sos_div_up(max_nt, 128);
    splits = sos_div_up(2 * ctx->sm_count, q_tiles * n_seg);
    if (splits > t_tiles / 4) splits = t_tiles / 4;
  } else {
    // split the train range so that a work item is ~256 x 1024 descriptor pairs and small problems still give every SM
    // several items; never finer than one shared-memory tile
    const int t_tiles = sos_div_up(max_nt > 0 ? max_nt : 1, HB_TILE_T);
    splits = sos_div_up(max_nt > 0 ? max_nt : 1, 1024);
    const int fill = sos_div_up(4 * ctx->sm_count, q_tiles * n_seg);
    if (splits < fill) splits = fill;
    if (splits > t_tiles) splits = t_tiles;
  }
  if (splits > (1 << ITEM_SPLIT_BITS)) splits = 1 << ITEM_SPLIT_BITS;
  if (splits < 1) splits = 1;

  void* ws = nullptr;
  const size_t rows_bound = (size_t)max_nq * (size_t)n_seg;
  const size_t max_items = (size_t)q_tiles * splits * n_seg;
  SOS_CHECK_ARG(max_items < ((size_t)1 << 31), "too many work items");
  const size_t partial_bytes = sos_align_up(rows_bound * splits * sizeof(uint2), 256);
  const size_t items_bytes = sos_align_up(max_items * sizeof(uint32_t), 256);
  const size_t exp_bytes = use_mma ? sos_hamming_mma_scratch_bytes(n_seg, max_nq, max_nt) : 0;
  int rc = sos_arena_get(ctx, partial_bytes + items_bytes + 256 + exp_bytes, &ws);
  if (rc != SOS_OK) return rc;
  uint32_t* items = (uint32_t*)((char*)ws + partial_bytes);
  int32_t* n_items = (int32_t*)((char*)ws + partial_bytes + items_bytes);

  hamming_plan_kernel<<<1, 256, 0, ctx->stream>>>(q_len, n_seg, max_nq, splits, items, n_items);
  SOS_LAUNCHED_AS(ctx, "hamming_plan_kernel");
  const unsigned grid = (unsigned)max_items;
  if (use_mma) {
    rc = sos_hamming_mma_launch(ctx, q, t, q_start, q_len, t_start, t_len, n_seg, max_nq, max_nt, splits, items, n_items,
                                grid, top2, (char*)ws + partial_bytes + items_bytes + 256, (uint2*)ws);
    if (rc != SOS_OK) return rc;
  } else {
#define HB_LAUNCH(T2)                                                                                                  \
  hamming_partial_kernel<T2><<<grid, HB_THREADS, 0, ctx->stream>>>((const uint4*)q, (const uint4*)t, q_start, q_len,    \
                                                                   t_start, t_len, max_nq, max_nt, splits, items,      \
                                                                   n_items, (uint2*)ws)
    if (top2) HB_LAUNCH(true); else HB_LAUNCH(false);
#undef HB_LAUNCH
    SOS_LAUNCHED_AS(ctx, "hamming_partial_kernel");
  }
  dim3 mgrid(sos_div_up(max_nq, 256), n_seg);
  hamming_merge_kernel<<<mgrid, 256, 0, ctx->stream>>>((const uint2*)ws, q_start, q_len, max_nq, splits, idx0, d0, idx1, d1);
  SOS_LAUNCHED_AS(ctx, "hamming_merge_kernel");
  return SOS_OK;
}

// ---------------------------------------------------------------------------------------------------
// radiusMatch: every train row within a descriptor distance of a query row.  One thread per query walks the train rows in
// index order (shared-memory tiles as above); pass 1 counts, pass 2 fills at the caller's offsets.  A non-default branch
// of FeatureMatcher.match (use_radius_match, camera_models.py:409-412): correctness first, no work splitting.
// ---------------------------------------------------------------------------------------------------
namespace {
template <bool FILL>
__global__ void __launch_bounds__(128)
hamming_radius_kernel(const uint4* __restrict__ q, int nq, const uint4* __restrict__ t, int nt, int max_dist,
                      int32_t* __restrict__ count, const int64_t* __restrict__ offset, int32_t* __restrict__ out_t,
                      int32_t* __restrict__ out_d) {
  __shared__ uint4 tile[HB_TILE_T * 2];
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = row < nq;
  uint4 qa = make_uint4(0, 0, 0, 0), qb = qa;
  if (live) { qa = __ldg(q + (size_t)row * 2); qb = __ldg(q + (size_t)row * 2 + 1); }
  int n = 0;
  int64_t base = FILL && live ? offset[row] : 0;
  for (int tb = 0; tb < nt; tb += HB_TILE_T) {
    const int n_tile = min(HB_TILE_T, nt - tb);
    __syncthreads();
    for (int i = threadIdx.x; i < n_tile * 2; i += blockDim.x) tile[i] = __ldg(t + (size_t)tb * 2 + i);
    __syncthreads();
    if (!live) continue;
    for (int j = 0; j < n_tile; ++j) {
      const uint4 ta = tile[j * 2], tbv = tile[j * 2 + 1];
      const int d = __popc(qa.x ^ ta.x) + __popc(qa.y ^ ta.y) + __popc(qa.z ^ ta.z) + __popc(qa.w ^ ta.w) +
                    __popc(qb.x ^ tbv.x) + __popc(qb.y ^ tbv.y) + __popc(qb.z ^ tbv.z) + __popc(qb.w ^ tbv.w);
      if (d <= max_dist) {
        if (FILL) { out_t[base + n] = tb + j; out_d[base + n] = d; }
        ++n;
      }
    }
  }
  if (!FILL && live) count[row] = n;
}
}  // namespace

extern "C" int sos_hamming_radius(sos_ctx* ctx, const uint32_t* q, int nq, const uint32_t* t, int nt, int max_distance,
                                  int32_t* count, const int64_t* offset, int32_t* out_t, int32_t* out_d) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(nq >= 0 && nt >= 0, "negative size");
  if (nq == 0) return SOS_OK;
  SOS_CHECK_ARG(q && (t || nt == 0), "NULL array");
  SOS_CHECK_ARG(((uintptr_t)q & 15) == 0 && ((uintptr_t)t & 15) == 0, "descriptor arrays must be 16-byte aligned");
  SOS_CHECK_ARG((count != nullptr) != (offset != nullptr), "pass either count (pass 1) or offset + out_t + out_d (pass 2)");
  SOS_CHECK_ARG(count || (out_t && out_d), "pass 2 needs out_t and out_d");
  SOS_CUDA(cudaSetDevice(ctx->device));
  const int grid = sos_div_up(nq, 128);
  if (count) hamming_radius_kernel<false><<<grid, 128, 0, ctx->stream>>>((const uint4*)q, nq, (const uint4*)t, nt, max_distance, count, nullptr, nullptr, nullptr);
  else hamming_radius_kernel<true><<<grid, 128, 0, ctx->stream>>>((const uint4*)q, nq, (const uint4*)t, nt, max_distance, nullptr, offset, out_t, out_d);
  SOS_LAUNCHED_AS(ctx, "hamming_radius_kernel");
  return SOS_OK;
}

// ---------------------------------------------------------------------------------------------------
// Float descriptors, L2 norm (cv2.BFMatcher() of the SIFT / SURF branch, camera_models.py:397-399): tensor-core engine only.
// ---------------------------------------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256)
l2_merge_kernel(const ulonglong2* __restrict__ partial, const int32_t* __restrict__ q_start, const int32_t* __restrict__ q_len,
                int max_nq, int splits, int32_t* __restrict__ idx0, float* __restrict__ d0, int32_t* __restrict__ idx1,
                float* __restrict__ d1) {
  const int seg = blockIdx.y;
  const int q0 = q_start[seg], nq = min(q_len[seg], max_nq);
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= nq) return;
  const ulonglong2* p = partial + ((size_t)seg * max_nq + row) * splits;
  unsigned long long k0 = ~0ull, k1 = ~0ull;
  for (int s = 0; s < splits; ++s) {
    const ulonglong2 v = p[s];
    k1 = min(k1, max(k0, v.x));
    k0 = min(k0, v.x);
    k1 = min(k1, v.y);
  }
  // cv2 reports sqrt of the float32 sum of squared differences; the sum is an exact integer < 2^24 here
  idx0[q0 + row] = (k0 == ~0ull) ? -1 : (int32_t)(k0 & 0xFFFFFFFFull);
  d0[q0 + row] = (k0 == ~0ull) ? -1.f : sqrtf((float)(uint32_t)(k0 >> 32));
  if (idx1) idx1[q0 + row] = (k1 == ~0ull) ? -1 : (int32_t)(k1 & 0xFFFFFFFFull);
  if (d1) d1[q0 + row] = (k1 == ~0ull) ? -1.f : sqrtf((float)(uint32_t)(k1 >> 32));
}
}  // namespace

extern "C" int sos_l2_top2(sos_ctx* ctx, const float* q, const float* t, int dim, const int32_t* q_start,
                           const int32_t* q_len, const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq,
                           int max_nt, int32_t* idx0, float* d0, int32_t* idx1, float* d1, int32_t* not_integer_flag) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n_seg >= 0 && max_nq >= 0 && max_nt >= 0, "negative size");
  SOS_CHECK_ARG(dim >= 1 && dim <= 128, "descriptor length must be 1..128 (SIFT: 128, SURF: 64)");
  SOS_CHECK_ARG(n_seg <= 65535, "at most 65535 segments per call");
  if (n_seg == 0 || max_nq == 0) return SOS_OK;
  SOS_CHECK_ARG(q && t && q_start && q_len && t_start && t_len && idx0 && d0 && not_integer_flag, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  const int q_tiles = sos_div_up(max_nq, HB_TILE_Q);
  SOS_CHECK_ARG(q_tiles <= (1 << ITEM_TILE_BITS), "segment has too many query rows (limit 262144)");
  const bool top2 = idx1 != nullptr || d1 != nullptr;
  const int t_tiles = sos_div_up(max_nt > 0 ? max_nt : 1, 128);
  int splits = sos_div_up(2 * ctx->sm_count, q_tiles * n_seg);
  if (splits > t_tiles / 4) splits = t_tiles / 4;
  if (splits > (1 << ITEM_SPLIT_BITS)) splits = 1 << ITEM_SPLIT_BITS;
  if (splits < 1) splits = 1;
  void* ws = nullptr;
  const size_t max_items = (size_t)q_tiles * splits * n_seg;
  SOS_CHECK_ARG(max_items < ((size_t)1 << 31), "too many work items");
  const size_t partial_bytes = sos_align_up((size_t)max_nq * n_seg * splits * sizeof(ulonglong2), 256);
  const size_t items_bytes = sos_align_up(max_items * sizeof(uint32_t), 256);
  int rc = sos_arena_get(ctx, partial_bytes + items_bytes + 256 + sos_l2_mma_scratch_bytes(n_seg, max_nq, max_nt), &ws);
  if (rc != SOS_OK) return rc;
  uint32_t* items = (uint32_t*)((char*)ws + partial_bytes);
  int32_t* n_items = (int32_t*)((char*)ws + partial_bytes + items_bytes);
  SOS_CUDA(cudaMemsetAsync(not_integer_flag, 0, sizeof(int32_t), ctx->stream));
  hamming_plan_kernel<<<1, 256, 0, ctx->stream>>>(q_len, n_seg, max_nq, splits, items, n_items);
  SOS_LAUNCHED_AS(ctx, "hamming_plan_kernel");
  rc = sos_l2_mma_launch(ctx, q, t, dim, q_start, q_len, t_start, t_len, n_seg, max_nq, max_nt, splits, items, n_items,
                         (unsigned)max_items, top2, (char*)ws + partial_bytes + items_bytes + 256, (ulonglong2*)ws,
                         not_integer_flag);
  if (rc != SOS_OK) return rc;
  dim3 mgrid(sos_div_up(max_nq, 256), n_seg);
  l2_merge_kernel<<<mgrid, 256, 0, ctx->stream>>>((const ulonglong2*)ws, q_start, q_len, max_nq, splits, idx0, d0, idx1, d1);
  SOS_LAUNCHED_AS(ctx, "l2_merge_kernel");
  return SOS_OK;
}

// Any finite float descriptors: the split-bfloat16 GEMM ranks, float64 decides (hamming_mma.cu: band, kernels).
extern "C" int sos_l2f_top2(sos_ctx* ctx, const float* q, const float* t, int dim, const int32_t* q_start,
                            const int32_t* q_len, const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq,
                            int max_nt, int32_t* idx0, float* d0, int32_t* idx1, float* d1, int32_t* nonfinite_flag,
                            int32_t* stats) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n_seg >= 0 && max_nq >= 0 && max_nt >= 0, "negative size");
  SOS_CHECK_ARG(dim >= 1 && dim <= 128, "descriptor length must be 1..128");
  SOS_CHECK_ARG(n_seg <= 65535, "at most 65535 segments per call");
  SOS_CHECK_ARG(max_nt < (1 << 30), "segment has too many train rows");
  if (n_seg == 0 || max_nq == 0) return SOS_OK;
  SOS_CHECK_ARG(q && t && q_start && q_len && t_start && t_len && idx0 && d0 && nonfinite_flag, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  const int q_tiles = sos_div_up(max_nq, HB_TILE_Q);
  SOS_CHECK_ARG(q_tiles <= (1 << ITEM_TILE_BITS), "segment has too many query rows (limit 262144)");
  const bool top2 = idx1 != nullptr || d1 != nullptr;
  const int t_tiles = sos_div_up(max_nt > 0 ? max_nt : 1, 128);
  int splits = sos_div_up(2 * ctx->sm_count, q_tiles * n_seg);
  if (splits > t_tiles / 4) splits = t_tiles / 4;
  if (splits > (1 << ITEM_SPLIT_BITS)) splits = 1 << ITEM_SPLIT_BITS;
  if (splits < 1) splits = 1;
  void* ws = nullptr;
  const size_t max_items = (size_t)q_tiles * splits * n_seg;
  SOS_CHECK_ARG(max_items < ((size_t)1 << 31), "too many work items");
  const size_t items_bytes = sos_align_up(max_items * sizeof(uint32_t), 256);
  int rc = sos_arena_get(ctx, items_bytes + 256 + sos_l2f_scratch_bytes(n_seg, max_nq, max_nt, dim, splits), &ws);
  if (rc != SOS_OK) return rc;
  uint32_t* items = (uint32_t*)ws;
  int32_t* n_items = (int32_t*)((char*)ws + items_bytes);
  SOS_CUDA(cudaMemsetAsync(nonfinite_flag, 0, sizeof(int32_t), ctx->stream));
  hamming_plan_kernel<<<1, 256, 0, ctx->stream>>>(q_len, n_seg, max_nq, splits, items, n_items);
  SOS_LAUNCHED_AS(ctx, "hamming_plan_kernel");
  return sos_l2f_launch(ctx, q, t, dim, q_start, q_len, t_start, t_len, n_seg, max_nq, max_nt, splits, items, n_items,
                        (unsigned)max_items, top2, (char*)ws + items_bytes + 256, idx0, d0, idx1, d1, nonfinite_flag, stats);
}

extern "C" int sos_match_select(sos_ctx* ctx, int mode, double ratio, const int32_t* idx0, const int32_t* d0,
                                const int32_t* d1, const int32_t* rev_idx0, const int32_t* q_start,
                                const int32_t* q_len, const int32_t* t_start, int n_seg, const float* px_q,
                                const float* px_t, double max_du, double min_dv, int32_t* out_q,
                                int32_t* out_t, int32_t* out_d, int32_t* out_count) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(mode == SOS_MATCH_NN || mode == SOS_MATCH_RATIO || mode == SOS_MATCH_CROSS, "unknown mode");
  SOS_CHECK_ARG(n_seg >= 0, "negative size");
  if (n_seg == 0) return SOS_OK;
  SOS_CHECK_ARG(idx0 && d0 && q_start && q_len && t_start && out_q && out_t && out_d && out_count, "NULL array");
  SOS_CHECK_ARG(mode != SOS_MATCH_RATIO || d1, "ratio mode needs d1");
  SOS_CHECK_ARG(mode != SOS_MATCH_CROSS || rev_idx0, "cross mode needs rev_idx0");
  SOS_CHECK_ARG((px_q == nullptr) == (px_t == nullptr), "px_q and px_t must be given together");
  SOS_CUDA(cudaSetDevice(ctx->device));
  SelectArgs a;
  a.mode = mode;
  a.ratio = ratio;
  a.idx0 = idx0; a.d0 = d0; a.d1 = d1; a.rev_idx0 = rev_idx0; a.q_start = q_start; a.q_len = q_len; a.t_start = t_start;
  a.px_q = (const float2*)px_q; a.px_t = (const float2*)px_t;
  a.max_du = max_du; a.min_dv = min_dv;
  a.out_q = out_q; a.out_t = out_t; a.out_d = out_d; a.out_count = out_count;
  match_select_kernel<<<n_seg, MS_THREADS, 0, ctx->stream>>>(a);
  SOS_LAUNCHED_AS(ctx, "match_select_kernel");
  return SOS_OK;
}

namespace {
__global__ void pixel_gate_kernel(const double2* __restrict__ top, const double2* __restrict__ bot, int n, double max_du,
                                  double min_dv, uint8_t* __restrict__ valid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double2 a = top[i], b = bot[i];
  bool ok = true;
  if (max_du > 0.0) ok = ok && (fabs(a.x - b.x) <= max_du);  // common_cv.py:177-178
  if (min_dv >= 0.0) ok = ok && (a.y - b.y >= min_dv);       // common_cv.py:182-184
  valid[i] = ok ? 1 : 0;
}
}  // namespace

extern "C" int sos_pixel_gate(sos_ctx* ctx, const double* pts_top, const double* pts_bot, int n, double max_du,
                              double min_dv, uint8_t* valid) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return SOS_OK;
  SOS_CHECK_ARG(pts_top && pts_bot && valid, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  pixel_gate_kernel<<<sos_div_up(n, 256), 256, 0, ctx->stream>>>((const double2*)pts_top, (const double2*)pts_bot, n, max_du,
                                                                  min_dv, valid);
  SOS_LAUNCHED_AS(ctx, "pixel_gate_kernel");
  return SOS_OK;
}
