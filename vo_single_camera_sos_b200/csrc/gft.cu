// Shi-Tomasi corner detection on the panoramas (SURVEY §8f row N3, detection half).
//
// replaces: cv2.goodFeaturesToTrack(image, maxCorners, qualityLevel = 0.01, minDistance = 5, mask = m,
//           useHarrisDetector = False) per azimuthal mask in OmniCamModel.detect_sparse_features_on_panorama
//           (camera_models.py:1737), i.e. cv::cornerMinEigenVal (blockSize 3, Sobel 3) + threshold at
//           quality * max over the mask + 3x3 non-maximum suppression + strongest-first minimum-distance selection.
//
// Arithmetic of cornerMinEigenVal, identified against cv2 (the tests restate it operation by operation in NumPy): Sobel in
// float32 with the scale s = 1/(4*3*255) folded into the smoothing taps.  dx: rows differentiated exactly, then smoothed
// down the column with one fused multiply-add, dx = fma(s, d[-1] + d[+1], 2s * d[0]).  dy: each row smoothed in tap order
// as cv2's row filter accumulates it, fma(s, g[x+1], fma(2s, g[x], s * g[x-1])), then the row above subtracted from the
// row below.  Covariance products in float32; the 3x3 box sums accumulate in float64 ((p[-1] + p[0]) + p[+1] along the
// row, then down the column) and are rounded once; eigenvalue (a + c) - sqrt((a - c)^2 + b^2) in float32 without
// contraction.  cv2 itself differs in its SIMD tail columns (the last <= 16 of a row, which skip the FMA) and, on sharp
// images, at a few interior pixels where its sliding-window box sums round differently (by at most half a unit of the
// image's largest measure).
//
// Selection: candidates of one (image, mask) are sorted by (strength desc, pixel index desc) — cv2's comparator — and the
// strongest-first greedy of cv2 is evaluated in parallel rounds (a candidate is accepted once every stronger candidate
// closer than minDistance has been rejected, rejected once one of them has been accepted): same result, no serial walk.
// Because a decision never depends on weaker candidates, only a histogram-picked prefix of the strongest candidates is sorted
// and decided, chunk by chunk, until maxCorners corners are accepted (whole list only if the prefix runs dry).
#include <math_constants.h>

#include <algorithm>
#include <vector>

#include "sos_common.cuh"

namespace {

__device__ __forceinline__ int refl(int p, int n) {
  if (n == 1) return 0;
  while (p < 0 || p >= n) p = p < 0 ? -p : 2 * n - 2 - p;
  return p;
}

// Corner measure + (optionally) the maximum over each mask, fused.  Per pixel: Sobel derivatives (cv2's arithmetic, see the
// top of the file), covariance terms dx^2, dx dy, dy^2 in float32, their 3 x 3 box sums in double (cv2's
// RowSum<float,double> / ColumnSum<double,float>), smaller eigenvalue without contraction.
// Every thread walks down its column with the 3-tap row sums of the last three rows in registers and recomputes the
// covariance terms of its three columns from the gray image, so nothing but the gray image is read and nothing but the
// measure is written.  (First version: a covariance image of 12 bytes per pixel written by one kernel and pulled through L2
// three times by the next - 0.34 + 0.89 ms for 32 C2 panoramas.)
// `mask_bits` holds one bit per mask and pixel; per warp only the masks present in the warp are reduced (one atomic per mask
// and warp at most).  Non-negative floats order like their bit patterns, so the maxima are kept as uint32.
constexpr int GE_ROWS = 16;   // rows per block

__global__ void __launch_bounds__(256, 3)
gft_eig_kernel(const uint8_t* __restrict__ gray, int H, int W, float* __restrict__ eig, const uint32_t* __restrict__ mask_bits,
               int n_masks, uint32_t* __restrict__ max_bits) {
  const int xr = blockIdx.x * blockDim.x + threadIdx.x, img = blockIdx.z;
  const int y0 = blockIdx.y * GE_ROWS, y1 = min(H, y0 + GE_ROWS);
  const bool in = xr < W;
  const int x = in ? xr : W - 1;
  const uint8_t* g = gray + (size_t)img * H * W;
  // the three columns whose covariance terms enter this pixel's box sums (BORDER_REFLECT_101), each with its own Sobel taps
  int cx[3][3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const int c0 = refl(x + j - 1, W);
    cx[j][0] = refl(c0 - 1, W);
    cx[j][1] = c0;
    cx[j][2] = refl(c0 + 1, W);
  }
  const float s = (float)(1.0 / (4.0 * 3.0 * 255.0)), s2 = 2.0f * s;
  double ha[3], hb[3], hc[3];
  auto row_sums = [&](int yy, double& a, double& b, double& cc) {
    const int yc = refl(yy, H);
    const uint8_t* ru = g + (size_t)refl(yc - 1, H) * W;
    const uint8_t* r0 = g + (size_t)yc * W;
    const uint8_t* rd = g + (size_t)refl(yc + 1, H) * W;
    float pxx[3], pxy[3], pyy[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const float a00 = ru[cx[j][0]], a01 = ru[cx[j][1]], a02 = ru[cx[j][2]];
      const float a10 = r0[cx[j][0]], a12 = r0[cx[j][2]];
      const float a20 = rd[cx[j][0]], a21 = rd[cx[j][1]], a22 = rd[cx[j][2]];
      const float du = a02 - a00, d0 = a12 - a10, dd = a22 - a20;
      const float dx = __fmaf_rn(s, du + dd, __fmul_rn(s2, d0));
      const float su = __fmaf_rn(s, a02, __fmaf_rn(s2, a01, __fmul_rn(s, a00)));
      const float sd = __fmaf_rn(s, a22, __fmaf_rn(s2, a21, __fmul_rn(s, a20)));
      const float dy = __fsub_rn(sd, su);
      pxx[j] = __fmul_rn(dx, dx);
      pxy[j] = __fmul_rn(dx, dy);
      pyy[j] = __fmul_rn(dy, dy);
    }
    a = ((double)pxx[0] + (double)pxx[1]) + (double)pxx[2];
    b = ((double)pxy[0] + (double)pxy[1]) + (double)pxy[2];
    cc = ((double)pyy[0] + (double)pyy[1]) + (double)pyy[2];
  };
  // Fast path (warp-uniform): no reflection anywhere in the strip.  Per gray row and column, D = g[x+1] - g[x-1] and
  // S = fma(s, g[x+1], fma(2s, g[x], s g[x-1])) are computed once and serve the three product rows that touch the row
  // (same operations, same order as the generic path: bit-identical).
  const bool fast = __all_sync(0xFFFFFFFFu, in && x >= 2 && x + 2 < W) && y0 >= 2 && y1 <= H - 2;
  float D[3][3], S[3][3];
  uint8_t raw[5];                                  // the gray row after next, loaded one iteration ahead of its use
  auto fetch = [&](int row) {
    const uint8_t* r = g + (size_t)min(row, H - 1) * W + (x - 2);
#pragma unroll
    for (int k = 0; k < 5; ++k) raw[k] = __ldg(r + k);
  };
  auto derive = [&](float* Dr, float* Sr) {
    float v[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) v[k] = raw[k];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      Dr[j] = v[j + 2] - v[j];
      Sr[j] = __fmaf_rn(s, v[j + 2], __fmaf_rn(s2, v[j + 1], __fmul_rn(s, v[j])));
    }
  };
  auto fast_sums = [&](double& a, double& b, double& cc) {
    float pxx[3], pxy[3], pyy[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const float dx = __fmaf_rn(s, D[0][j] + D[2][j], __fmul_rn(s2, D[1][j]));
      const float dy = __fsub_rn(S[2][j], S[0][j]);
      pxx[j] = __fmul_rn(dx, dx);
      pxy[j] = __fmul_rn(dx, dy);
      pyy[j] = __fmul_rn(dy, dy);
    }
    a = ((double)pxx[0] + (double)pxx[1]) + (double)pxx[2];
    b = ((double)pxy[0] + (double)pxy[1]) + (double)pxy[2];
    cc = ((double)pyy[0] + (double)pyy[1]) + (double)pyy[2];
  };
  auto shift = [&]() {
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      D[0][j] = D[1][j]; D[1][j] = D[2][j];
      S[0][j] = S[1][j]; S[1][j] = S[2][j];
    }
  };
  if (fast) {
    fetch(y0 - 2); derive(D[0], S[0]);
    fetch(y0 - 1); derive(D[1], S[1]);
    fetch(y0);     derive(D[2], S[2]);
    fast_sums(ha[0], hb[0], hc[0]);
    shift();
    fetch(y0 + 1); derive(D[2], S[2]);
    fast_sums(ha[1], hb[1], hc[1]);
    fetch(y0 + 2);
  } else {
    row_sums(y0 - 1, ha[0], hb[0], hc[0]);
    row_sums(y0, ha[1], hb[1], hc[1]);
  }
  uint32_t tm = 0u, tv = 0u;                      // tracked mask set and the largest measure (as bits) seen under it
  auto flush = [&]() {
    uint32_t present = __reduce_or_sync(0xFFFFFFFFu, tm);
    while (present) {
      const int m = __ffs(present) - 1;
      present &= present - 1;
      const uint32_t best = __reduce_max_sync(0xFFFFFFFFu, ((tm >> m) & 1u) ? tv : 0u);
      if ((threadIdx.x & 31) == 0 && best > 0u) atomicMax(&max_bits[img * n_masks + m], best);
    }
    tm = 0u;
    tv = 0u;
  };
  for (int y = y0; y < y1; ++y) {
    const uint32_t mb_next = (mask_bits && in) ? __ldg(&mask_bits[(size_t)y * W + x]) : 0u;   // early: overlaps the arithmetic
    if (fast) {
      shift();
      derive(D[2], S[2]);                          // gray row y + 2
      fetch(y + 3);
      fast_sums(ha[2], hb[2], hc[2]);
    } else {
      row_sums(y + 1, ha[2], hb[2], hc[2]);
    }
    const double sa = (ha[0] + ha[1]) + ha[2], sb = (hb[0] + hb[1]) + hb[2], sc = (hc[0] + hc[1]) + hc[2];
    ha[0] = ha[1]; ha[1] = ha[2];
    hb[0] = hb[1]; hb[1] = hb[2];
    hc[0] = hc[1]; hc[1] = hc[2];
    const float a = __fmul_rn((float)sa, 0.5f), b = (float)sb, cc = __fmul_rn((float)sc, 0.5f);
    const float t = __fsub_rn(a, cc);
    const float r = __fsqrt_rn(__fadd_rn(__fmul_rn(t, t), __fmul_rn(b, b)));
    const float v = __fsub_rn(__fadd_rn(a, cc), r);
    if (in) eig[((size_t)img * H + y) * W + x] = v;
    if (mask_bits) {
      // running maximum per thread while its mask set stays the same down the column (the usual case: masks are column
      // ranges); the warp flushes to the global maxima when some lane's set changes and at the end of the strip - a
      // global read-compare-atomic per row would put an L2 round trip into every iteration of the walk
      const uint32_t mb = (in && v > 0.f) ? mb_next : 0u;
      if (__any_sync(0xFFFFFFFFu, mb != 0u && tm != 0u && mb != tm)) flush();
      if (mb) {
        tm = mb;
        tv = max(tv, __float_as_uint(v));
      }
    }
  }
  if (mask_bits) flush();
}

// one bit per mask and pixel (masks are shared by all images); flags pixels that belong to more than one mask
__global__ void gft_pack_masks_kernel(const uint8_t* __restrict__ masks, size_t per, int n_masks, uint32_t* __restrict__ bits,
                                      int32_t* __restrict__ overlap) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= per) return;
  uint32_t b = 0;
  if (!masks) b = 1u;
  else
    for (int m = 0; m < n_masks; ++m) b |= (masks[(size_t)m * per + i] ? 1u : 0u) << m;
  bits[i] = b;
  if (__popc(b) > 1) *overlap = 1;
}

// candidates: interior pixels above the mask's threshold that equal the maximum of their 3x3 neighbourhood.
// A block covers GC_ROWS rows x 256 columns, stages its candidates in shared memory and reserves their slots in the
// per-list arrays with ONE global atomic per (block, mask): returning atomics on a few hundred hot counters were the whole
// cost of the first version (ncu: long-scoreboard stall 94, every pipe idle).
constexpr int GC_ROWS = 8;
constexpr int GC_STAGE = 1024;

__global__ void __launch_bounds__(256)
gft_candidates_kernel(const float* __restrict__ eig, const uint32_t* __restrict__ mask_bits, int H, int W, int n_masks,
                      const uint32_t* __restrict__ max_bits, double quality, int cap, unsigned long long* __restrict__ keys,
                      int32_t* __restrict__ counts) {
  __shared__ unsigned long long s_key[GC_STAGE];
  __shared__ uint8_t s_m[GC_STAGE];
  __shared__ int s_n, s_cnt[32], s_base[32], s_fill[32];
  __shared__ float s_thr[32];
  const int x = blockIdx.x * blockDim.x + threadIdx.x, img = blockIdx.z;
  if (threadIdx.x < 32) {
    s_cnt[threadIdx.x] = 0;
    s_fill[threadIdx.x] = 0;
    // threshold(eig, eig, maxVal * qualityLevel, 0, THRESH_TOZERO) with the mask's own maximum
    s_thr[threadIdx.x] = threadIdx.x < n_masks ? (float)((double)__uint_as_float(max_bits[img * n_masks + threadIdx.x]) * quality)
                                               : CUDART_INF_F;
  }
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  const float* e = eig + (size_t)img * H * W;
  for (int r = 0; r < GC_ROWS; ++r) {
    const int y = blockIdx.y * GC_ROWS + r;
    if (x < 1 || x >= W - 1 || y < 1 || y >= H - 1) continue;
    const size_t px = (size_t)y * W + x;
    const float v = e[px];
    if (!(v > 0.f)) continue;
    uint32_t mb = mask_bits[px], pass = 0;
    while (mb) {                                         // the threshold test first: one load, removes most pixels
      const int m = __ffs(mb) - 1;
      mb &= mb - 1;
      if (v > s_thr[m]) pass |= 1u << m;
    }
    if (!pass) continue;
    float nb = 0.f;
#pragma unroll
    for (int j = -1; j <= 1; ++j)
#pragma unroll
      for (int i = -1; i <= 1; ++i) nb = fmaxf(nb, e[(size_t)(y + j) * W + x + i]);
    if (v != nb) continue;
    const unsigned long long key = ((unsigned long long)__float_as_uint(v) << 32) | (uint32_t)px;
    while (pass) {
      const int m = __ffs(pass) - 1;
      pass &= pass - 1;
      const int i = atomicAdd(&s_n, 1);
      if (i < GC_STAGE) {
        s_key[i] = key;
        s_m[i] = (uint8_t)m;
        atomicAdd(&s_cnt[m], 1);
      } else {                                           // staging full (cannot happen with 3x3 maxima on 8 x 256 pixels)
        const int slot = atomicAdd(&counts[img * n_masks + m], 1);
        if (slot < cap) keys[((size_t)(img * n_masks + m)) * cap + slot] = key;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < n_masks && s_cnt[threadIdx.x] > 0)
    s_base[threadIdx.x] = atomicAdd(&counts[img * n_masks + threadIdx.x], s_cnt[threadIdx.x]);
  __syncthreads();
  const int n = min(s_n, GC_STAGE);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int m = s_m[i];
    const int slot = s_base[m] + atomicAdd(&s_fill[m], 1);
    if (slot < cap) keys[((size_t)(img * n_masks + m)) * cap + slot] = s_key[i];
  }
}

constexpr int GFT_CAP = 16384;      // candidates per (image, mask) kept for the selection (128 KB of shared memory)
constexpr int GFT_THREADS = 1024;
constexpr int GFT_K = 4;            // stronger neighbours remembered per candidate (more: rescan the rank image)

constexpr int GFT_CHUNK = 2048;     // candidates decided per pass of the selection (strongest first)

// Shared memory of the selection for a list sorted as np2 keys: keys, one state byte per candidate, and the neighbour lists of
// one chunk.
__host__ __device__ inline size_t gft_select_smem(int np2) {
  return (size_t)np2 * (sizeof(unsigned long long) + 1) + (size_t)GFT_CHUNK * (GFT_K * sizeof(uint16_t) + 1);
}

// One block per (image, mask): sort descending, then cv2's strongest-first minimum-distance greedy.  A candidate's fate only
// depends on STRONGER candidates, so the sorted list is decided chunk by chunk (parallel rounds inside a chunk) and the
// kernel stops as soon as max_corners corners are accepted - usually inside the first chunk or two.
__global__ void __launch_bounds__(GFT_THREADS)
gft_select_kernel(const unsigned long long* __restrict__ keys_in, const int32_t* __restrict__ counts, int cap, int H, int W,
                  int n_masks, int mask_index, int max_corners, int min_dist_sq, int reach, int32_t* __restrict__ rank_img,
                  float* __restrict__ out_xy, int32_t* __restrict__ out_count) {
  extern __shared__ unsigned long long skey[];
  __shared__ int n_undecided, s_fill, s_bin;
  __shared__ uint32_t s_maxhi;
  __shared__ int warp_sums[GFT_THREADS / 32];
  // mask_index >= 0: one launch per mask (masks may overlap, the rank image of an image serves one mask at a time);
  // mask_index < 0: masks are pixel-disjoint, one launch for all lists, rank-image entries are tagged with their mask
  const int img = mask_index >= 0 ? blockIdx.x : blockIdx.x / n_masks;
  const int mk = mask_index >= 0 ? mask_index : blockIdx.x % n_masks;
  const int list = img * n_masks + mk;
  const int tag = mk << 16;
  if (counts[list] > cap) {
    // more local maxima than the candidate buffer holds (the host refuses the call before launching; this keeps the
    // kernel inside its shared memory whatever it is given)
    if (threadIdx.x == 0) out_count[list] = -counts[list];
    return;
  }
  const int n = counts[list];
  int np2 = 8;                                                // >= 8 keeps the byte / uint16 arrays behind the keys aligned
  while (np2 < n) np2 <<= 1;
  uint8_t* state = (uint8_t*)(skey + np2);                    // 0 undecided, 1 accepted, 2 rejected
  uint16_t* nbr = (uint16_t*)(state + np2);                   // [GFT_CHUNK][GFT_K] stronger neighbours of the chunk's candidates
  uint8_t* ncnt = (uint8_t*)(nbr + (size_t)GFT_CHUNK * GFT_K);
  const unsigned long long* kin = keys_in + (size_t)list * cap;
  int32_t* rimg = rank_img + (size_t)img * H * W;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // Only the strongest few thousand candidates can matter (the walk stops at max_corners accepted), and the sort is the
  // expensive part (a 16 K bitonic sort is 105 passes), so a histogram of the strength bits first picks a prefix of about
  // 4 max_corners candidates to sort and decide; if that prefix runs dry the whole list is sorted and the walk starts over.
  const int target = min(n, max(1024, 4 * max_corners));
  const bool preselect = min_dist_sq > 0 && n > 2 * target;
  int ns = n, processed = 0, accepted = 0;
  for (int attempt = 0; attempt < 2; ++attempt) {
    if (preselect && attempt == 0) {
      uint32_t* hist = (uint32_t*)nbr;                          // 1024 bins, free until the first chunk
      if (threadIdx.x == 0) { s_maxhi = 0u; s_fill = 0; }
      for (int i = threadIdx.x; i < 1024; i += blockDim.x) hist[i] = 0u;
      __syncthreads();
      uint32_t mh = 0u;
      for (int i = threadIdx.x; i < n; i += blockDim.x) mh = max(mh, (uint32_t)(kin[i] >> 32));
      mh = __reduce_max_sync(0xFFFFFFFFu, mh);
      if (lane == 0) atomicMax(&s_maxhi, mh);
      __syncthreads();
      const uint32_t maxhi = s_maxhi;
      for (int i = threadIdx.x; i < n; i += blockDim.x) atomicAdd(&hist[min(1023u, (maxhi - (uint32_t)(kin[i] >> 32)) >> 16)], 1u);
      __syncthreads();
      if (warp == 0) {
        uint32_t loc = 0u;
        for (int q = 0; q < 32; ++q) loc += hist[lane * 32 + q];
        uint32_t inc = loc;
  #pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, off);
          if (lane >= off) inc += t;
        }
        const unsigned ball = __ballot_sync(0xFFFFFFFFu, inc >= (uint32_t)target);   // never empty: the bins hold all n >= target
        if (lane == __ffs(ball) - 1) {
          uint32_t cum = inc - loc;
          for (int q = 0; q < 32; ++q) {
            cum += hist[lane * 32 + q];
            if (cum >= (uint32_t)target) { s_bin = lane * 32 + q; break; }
          }
        }
      }
      __syncthreads();
      const uint32_t last_bin = (uint32_t)s_bin;
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const unsigned long long k = kin[i];
        if (min(1023u, (maxhi - (uint32_t)(k >> 32)) >> 16) <= last_bin) skey[atomicAdd(&s_fill, 1)] = k;
      }
      __syncthreads();
      ns = s_fill;
    } else {
      for (int i = threadIdx.x; i < n; i += blockDim.x) skey[i] = kin[i];
      ns = n;
    }
    int nps = 1;
    while (nps < ns) nps <<= 1;
    for (int i = ns + threadIdx.x; i < nps; i += blockDim.x) skey[i] = 0ull;
    __syncthreads();
    // bitonic sort, descending (key = strength bits << 32 | pixel index: cv2's greaterThanPtr order)
    for (int k = 2; k <= nps; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = threadIdx.x; i < nps; i += blockDim.x) {
          const int l = i ^ j;
          if (l > i) {
            const unsigned long long a = skey[i], b = skey[l];
            const bool desc = (i & k) == 0;
            if (desc ? (a < b) : (a > b)) { skey[i] = b; skey[l] = a; }
          }
        }
        __syncthreads();
      }
    processed = 0;
    accepted = 0;
    if (min_dist_sq > 0) {
      while (processed < ns && accepted < max_corners) {
        const int c0 = processed, c1 = min(ns, c0 + GFT_CHUNK);
        for (int i = c0 + threadIdx.x; i < c1; i += blockDim.x) {
          rimg[(uint32_t)skey[i]] = tag | i;
          state[i] = 0;
        }
        __syncthreads();
        // phase A: the stronger candidates closer than minDistance to candidate i.  All rank-image loads of a candidate are
        // independent, so they overlap; the rounds below then touch only these few shared-memory entries.
        for (int i = c0 + threadIdx.x; i < c1; i += blockDim.x) {
          const int px = (int)(uint32_t)skey[i];
          const int y = px / W, x = px - y * W;
          int cnt = 0;
          for (int dy = -reach; dy <= reach; ++dy) {
            const int yy = y + dy;
            if (yy < 0 || yy >= H) continue;
            for (int dx = -reach; dx <= reach; ++dx) {
              const int xx = x + dx;
              if (xx < 0 || xx >= W || dx * dx + dy * dy >= min_dist_sq) continue;
              const int e = rimg[(size_t)yy * W + xx];
              const int j = e & 0xFFFF;
              if (e >= 0 && (e >> 16) == mk && j < i) {
                if (cnt < GFT_K) nbr[(size_t)(i - c0) * GFT_K + cnt] = (uint16_t)j;
                ++cnt;
              }
            }
          }
          ncnt[i - c0] = (uint8_t)min(cnt, 255);
          if (cnt == 0) state[i] = 1;            // nothing stronger nearby: accepted outright
        }
        // phase B: rounds over the chunk's undecided candidates
        while (true) {
          __syncthreads();
          if (threadIdx.x == 0) n_undecided = 0;
          __syncthreads();
          int still = 0;
          for (int i = c0 + threadIdx.x; i < c1; i += blockDim.x) {
            if (state[i] != 0) continue;
            bool rejected = false, wait = false;
            const int cnt = ncnt[i - c0];
            if (cnt <= GFT_K) {
              for (int q = 0; q < cnt; ++q) {
                const uint8_t sj = ((volatile uint8_t*)state)[nbr[(size_t)(i - c0) * GFT_K + q]];
                if (sj == 1) { rejected = true; break; }
                if (sj == 0) wait = true;
              }
            } else {                              // more neighbours than the list holds (plateaus): rescan the rank image
              const int px = (int)(uint32_t)skey[i];
              const int y = px / W, x = px - y * W;
              for (int dy = -reach; dy <= reach && !rejected; ++dy) {
                const int yy = y + dy;
                if (yy < 0 || yy >= H) continue;
                for (int dx = -reach; dx <= reach; ++dx) {
                  const int xx = x + dx;
                  if (xx < 0 || xx >= W || dx * dx + dy * dy >= min_dist_sq) continue;
                  const int e = rimg[(size_t)yy * W + xx];
                  const int j = e & 0xFFFF;
                  if (e < 0 || (e >> 16) != mk || j >= i) continue;
                  const uint8_t sj = ((volatile uint8_t*)state)[j];
                  if (sj == 1) { rejected = true; break; }
                  if (sj == 0) wait = true;
                }
              }
            }
            // a decision only depends on FINAL states of stronger candidates, so the evaluation order inside a round is free
            if (rejected) ((volatile uint8_t*)state)[i] = 2;
            else if (!wait) ((volatile uint8_t*)state)[i] = 1;
            else ++still;
          }
          if (still) atomicAdd(&n_undecided, still);
          __syncthreads();
          if (n_undecided == 0) break;
        }
        for (int i0 = c0; i0 < c1; i0 += blockDim.x) {
          const int i = i0 + threadIdx.x;
          accepted += __syncthreads_count(i < c1 && state[i] == 1);
        }
        processed = c1;
      }
    } else {
      processed = min(n, max_corners);
      for (int i = threadIdx.x; i < processed; i += blockDim.x) state[i] = 1;
      __syncthreads();
    }
    if (!(preselect && attempt == 0 && accepted < max_corners && ns < n)) break;
    // the prefix ran dry: take the rank image back and decide the whole list
    for (int i = threadIdx.x; i < processed; i += blockDim.x) rimg[(uint32_t)skey[i]] = -1;
    __syncthreads();
  }
  // ordered compaction of the accepted candidates, at most max_corners
  int base = 0;
  for (int i0 = 0; i0 < processed && base < max_corners; i0 += blockDim.x) {
    const int i = i0 + threadIdx.x;
    const bool acc = i < processed && state[i] == 1;
    const unsigned vote = __ballot_sync(0xFFFFFFFFu, acc);
    if (lane == 0) warp_sums[warp] = __popc(vote);
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < GFT_THREADS / 32; ++w) {
      const int c = warp_sums[w];
      if (w < warp) before += c;
      total += c;
    }
    if (acc) {
      const int pos = base + before + __popc(vote & ((1u << lane) - 1u));
      if (pos < max_corners) {
        const int px = (int)(uint32_t)skey[i];
        const int y = px / W, x = px - y * W;
        out_xy[((size_t)list * max_corners + pos) * 2 + 0] = (float)x;
        out_xy[((size_t)list * max_corners + pos) * 2 + 1] = (float)y;
      }
    }
    base += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) out_count[list] = min(base, max_corners);
  // leave the rank image clean for the next mask / call
  if (min_dist_sq > 0)
    for (int i = threadIdx.x; i < processed; i += blockDim.x) rimg[(uint32_t)skey[i]] = -1;
}

}  // namespace

extern "C" int sos_corner_min_eigenval(sos_ctx* ctx, const uint8_t* gray, int n_images, int height, int width, float* eig) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n_images >= 0 && height >= 0 && width >= 0, "negative size");
  if (n_images == 0 || height == 0 || width == 0) return SOS_OK;
  SOS_CHECK_ARG(gray && eig, "NULL array");
  SOS_CHECK_ARG(n_images <= 65535 && height <= 65535, "too many images / rows");
  SOS_CUDA(cudaSetDevice(ctx->device));
  gft_eig_kernel<<<dim3(sos_div_up(width, 256), sos_div_up(height, GE_ROWS), n_images), 256, 0, ctx->stream>>>(gray, height, width, eig, nullptr, 0,
                                                                                                                 nullptr);
  SOS_LAUNCHED_AS(ctx, "gft_eig_kernel");
  return SOS_OK;
}

extern "C" int sos_gft_detect(sos_ctx* ctx, const uint8_t* gray, const uint8_t* masks, int n_images, int height, int width,
                              int n_masks, int max_corners, double quality_level, double min_distance, float* out_xy,
                              int32_t* out_count, float* eig_out) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n_images >= 0 && height >= 0 && width >= 0 && n_masks >= 1 && n_masks <= 32, "bad size (at most 32 masks)");
  // cv2 reads maxCorners <= 0 as "no limit"; here it sizes out_xy, so a limit is required
  SOS_CHECK_ARG(max_corners >= 1, "max_corners must be >= 1");
  SOS_CHECK_ARG(quality_level > 0.0 && min_distance >= 0.0 && min_distance < 64.0, "bad quality level / minimum distance");
  if (n_images == 0) return SOS_OK;
  SOS_CHECK_ARG(gray && out_count && out_xy, "NULL array");
  SOS_CHECK_ARG(height >= 3 && width >= 3 && (size_t)height * width < (1ull << 31), "image size out of range");
  SOS_CHECK_ARG((long long)n_images * n_masks <= 65535, "too many (image, mask) lists");
  SOS_CUDA(cudaSetDevice(ctx->device));
  const size_t px = (size_t)n_images * height * width;
  const int lists = n_images * n_masks;
  // scratch layout
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += sos_align_up(bytes, 256); return o; };
  const size_t o_eig = take(px * sizeof(float));
  const size_t o_max = take((size_t)lists * sizeof(uint32_t));
  const size_t o_cnt = take((size_t)lists * sizeof(int32_t));
  const size_t o_keys = take((size_t)lists * GFT_CAP * sizeof(unsigned long long));
  const size_t o_rank = take(px * sizeof(int32_t));
  const size_t o_flag = take(sizeof(int32_t));
  const size_t o_bits = take((size_t)height * width * sizeof(uint32_t));
  void* ws = nullptr;
  const int rc = sos_arena_get(ctx, off, &ws);
  if (rc != SOS_OK) return rc;
  uint8_t* base = (uint8_t*)ws;
  float* eig = (float*)(base + o_eig);
  uint32_t* max_bits = (uint32_t*)(base + o_max);
  int32_t* counts = (int32_t*)(base + o_cnt);
  unsigned long long* keys = (unsigned long long*)(base + o_keys);
  int32_t* rank_img = (int32_t*)(base + o_rank);

  dim3 grid(sos_div_up(width, 256), height, n_images);
  const size_t per = (size_t)height * width;
  uint32_t* mask_bits = (uint32_t*)(base + o_bits);
  int32_t* flag = (int32_t*)(base + o_flag);
  SOS_CUDA(cudaMemsetAsync(base + o_max, 0, (o_keys - o_max), ctx->stream));          // max_bits and counts
  SOS_CUDA(cudaMemsetAsync(flag, 0, sizeof(int32_t), ctx->stream));
  SOS_CUDA(cudaMemsetAsync(rank_img, 0xFF, px * sizeof(int32_t), ctx->stream));       // -1
  gft_pack_masks_kernel<<<(unsigned)((per + 255) / 256), 256, 0, ctx->stream>>>(masks, per, n_masks, mask_bits, flag);
  SOS_LAUNCHED_AS(ctx, "gft_pack_masks_kernel");
  gft_eig_kernel<<<dim3(grid.x, sos_div_up(height, GE_ROWS), grid.z), 256, 0, ctx->stream>>>(gray, height, width, eig, mask_bits, n_masks, max_bits);
  SOS_LAUNCHED_AS(ctx, "gft_eig_kernel");
  if (eig_out) SOS_CUDA(cudaMemcpyAsync(eig_out, eig, px * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
  gft_candidates_kernel<<<dim3(sos_div_up(width, 256), sos_div_up(height, GC_ROWS), n_images), 256, 0, ctx->stream>>>(
      eig, mask_bits, height, width, n_masks, max_bits, quality_level, GFT_CAP, keys, counts);
  SOS_LAUNCHED_AS(ctx, "gft_candidates_kernel");
  const size_t smem = gft_select_smem(GFT_CAP);
  // per device, so set on every call (a process may hold contexts on several devices)
  SOS_CUDA(cudaFuncSetAttribute(gft_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const double md2 = min_distance * min_distance;
  const int min_dist_sq = min_distance >= 1.0 ? (int)ceil(md2) : 0;   // integer offsets: dx^2 + dy^2 < minDistance^2
  const int reach = (int)ceil(min_distance);
  // One small read-back on every call: the overlap flag and the candidate counts.  A list with more candidates than the
  // buffer holds is refused (the atomics that filled the buffer kept a schedule-dependent subset), and the largest count
  // sizes the selection's shared memory (a block sorts next_pow2(count) keys: 64 KB instead of 128 KB lets three blocks
  // share an SM).
  int overlap = 0;
  std::vector<int32_t> hc(lists);
  SOS_CUDA(cudaMemcpyAsync(&overlap, flag, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  SOS_CUDA(cudaMemcpyAsync(hc.data(), counts, sizeof(int32_t) * lists, cudaMemcpyDeviceToHost, ctx->stream));
  SOS_CUDA(cudaStreamSynchronize(ctx->stream));
  int mx = 1;
  for (int v : hc) {
    if (v > GFT_CAP) {
      sos_set_error("sos_gft_detect: %d corner candidates in one mask, the selection holds %d: raise quality_level", v, GFT_CAP);
      return SOS_ERR_INVALID;
    }
    mx = std::max(mx, v);
  }
  int np2 = 1024;
  while (np2 < mx) np2 <<= 1;
  const size_t sel_smem = gft_select_smem(np2);
  // pixel-disjoint masks (the reference's default, overlap_degrees = 0): every list at once.  Overlapping masks: a pixel can
  // be a candidate of two lists and each selection needs the rank image of its image to itself -> one launch per mask.
  if (!overlap) {
    gft_select_kernel<<<lists, GFT_THREADS, sel_smem, ctx->stream>>>(keys, counts, GFT_CAP, height, width, n_masks, -1, max_corners,
                                                                 min_dist_sq, reach, rank_img, out_xy, out_count);
    SOS_LAUNCHED_AS(ctx, "gft_select_kernel");
    return SOS_OK;
  }
  for (int m = 0; m < n_masks; ++m) {
    gft_select_kernel<<<n_images, GFT_THREADS, sel_smem, ctx->stream>>>(keys, counts, GFT_CAP, height, width, n_masks, m, max_corners,
                                                                    min_dist_sq, reach, rank_img, out_xy, out_count);
    SOS_LAUNCHED_AS(ctx, "gft_select_kernel");
  }
  return SOS_OK;
}
