// Shared by the descriptor matchers: hamming.cu (C-ABI entry points, XOR+POPC engine) and hamming_mma.cu (tensor-core
// engines).  The work-item list, the partial-key formats, the planning and merge kernels, and the one host path of the
// three tensor-core engines.
#pragma once
#include "sos_common.cuh"
#include "tc_common.cuh"

// Work list: segment lengths live on the device, so the host can only size the grid for the worst case.  Launching
// that grid directly leaves the SMs unevenly loaded (blocks of short segments exit at once and everything fits in
// one wave: measured 66 % average SM activity).  Instead one small block compacts the ACTIVE (segment, query tile,
// train split) items into a list; block i of the matching kernel takes item i, so the active blocks are contiguous in
// launch order and the hardware scheduler balances them.
constexpr int ITEM_QROWS = 256;                          // query rows per work item
constexpr int ITEM_SPLIT_BITS = 6, ITEM_TILE_BITS = 10;  // item = seg << 16 | query tile << 6 | split

// Hamming partial key: distance << KEY_IDX_BITS | train row of the segment, so that min / max on the key give OpenCV's
// (distance, lowest index) order.  Up to 4M train rows per segment; distance <= 256 needs 9 bits.
constexpr int KEY_IDX_BITS = 22;
constexpr uint32_t KEY_NONE = 0xFFFFFFFFu;

namespace {

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
    const int tiles = seg < n_seg ? (min(q_len[seg], max_nq) + ITEM_QROWS - 1) / ITEM_QROWS : 0;
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

// (index, distance) of a partial key; all ones = none
__device__ __forceinline__ void key_decode(uint32_t k, int32_t& idx, int32_t& d) {   // Hamming
  idx = (k == KEY_NONE) ? -1 : (int32_t)(k & ((1u << KEY_IDX_BITS) - 1u));
  d = (k == KEY_NONE) ? -1 : (int32_t)(k >> KEY_IDX_BITS);
}
__device__ __forceinline__ void key_decode(unsigned long long k, int32_t& idx, float& d) {   // L2: squared distance << 32 | row
  idx = (k == ~0ull) ? -1 : (int32_t)(k & 0xFFFFFFFFull);
  // cv2 reports sqrt of the float32 sum of squared differences; the sum is an exact integer < 2^24 here
  d = (k == ~0ull) ? -1.f : sqrtf((float)(uint32_t)(k >> 32));
}

// One thread per query row: merge the per-split sorted key pairs (Pair = uint2: Hamming keys, ulonglong2: L2 keys)
template <typename Pair, typename Dist>
__global__ void __launch_bounds__(256)
merge_kernel(const Pair* __restrict__ partial, const int32_t* __restrict__ q_start, const int32_t* __restrict__ q_len,
             int max_nq, int splits, int32_t* __restrict__ idx0, Dist* __restrict__ d0, int32_t* __restrict__ idx1,
             Dist* __restrict__ d1) {
  using Key = decltype(Pair::x);
  const int seg = blockIdx.y;
  const int q0 = q_start[seg], nq = min(q_len[seg], max_nq);
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= nq) return;
  const Pair* p = partial + ((size_t)seg * max_nq + row) * splits;
  Key k0 = ~(Key)0, k1 = ~(Key)0;
  for (int s = 0; s < splits; ++s) {
    const Pair v = p[s];
    // merge two sorted pairs: v.x <= v.y
    k1 = min(k1, max(k0, v.x));
    k0 = min(k0, v.x);
    k1 = min(k1, v.y);  // v.y >= v.x, so it can only compete for second place
  }
  int32_t i;
  Dist d;
  key_decode(k0, i, d);
  idx0[q0 + row] = i;
  d0[q0 + row] = d;
  key_decode(k1, i, d);
  if (idx1) idx1[q0 + row] = i;
  if (d1) d1[q0 + row] = d;
}

}  // namespace

// The tensor-core engines (hamming_mma.cu) behind sos_hamming_top2 (KIND_HAMMING: q, t are 256-bit descriptors, d0 / d1
// int32), sos_l2_top2 (KIND_L2) and sos_l2f_top2 (KIND_L2F: q, t are float rows of length dim, d0 / d1 float).  Arguments are
// checked by the caller; flag is the caller's cleared not-integer / non-finite flag, stats the optional L2F statistics.
int sos_tc_match(sos_ctx* ctx, int kind, const void* q, const void* t, int dim, const int32_t* q_start, const int32_t* q_len,
                 const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq, int max_nt, int32_t* idx0, void* d0,
                 int32_t* idx1, void* d1, int32_t* flag, int32_t* stats);
