// Tensor-core engine of the RANSAC scores (step 5 of the SOS front-end): the reference's bearing-angle score, and the
// Euclidean score of the 3D-3D stress configuration (end of this comment).  Included by ransac.cu inside its anonymous namespace, after HypRec / Rig / ScoreConst / decision / guard_of / inlier_exact.
//
// The score of (hypothesis h, correspondence j) is  1 - f_j . x / |x| < thr  with  x = A_h p_j + b_h  (per camera; reference
// omnistereo/pose_est_tools.py:150-203 with the non-central correction of its comment at :181-185).  Both quantities the
// decision needs are BILINEAR in (hypothesis, correspondence) features:
//     s  = f . x  = sum_ik A_ik (f_i p_k) + sum_i b_i f_i                                        12 terms
//     n2 = |x|^2  = sum_kl (A^T A)_kl p_k p_l + 2 sum_k (A^T b)_k p_k + |b|^2                     10 terms
// i.e. two small-K GEMMs over (hypotheses x correspondences), and the decision is  D = s |s| - (1 - thr)^2 n2 > 0.
// The FP32 kernel (score_kernel) spends 19 FMA-pipe lanes per pair on them; here they come out of the 5th-generation
// tensor cores and the SM's ALUs only see 4 instructions per pair:
//   * every float32 feature is split exactly into three bfloat16 pieces (8 + 8 + 8 mantissa bits), and the six partial
//     products hi*hi, hi*mid, mid*hi, hi*lo, lo*hi, mid*mid are laid out as six K columns per feature (what is dropped is
//     below 2^-25 of the term), so a tcgen05.mma kind::f16 with float32 accumulators in tensor memory reproduces the
//     float32 product to ~1e-7 relative; K = 13*6 -> 80 columns for s (the thirteenth feature serves the Euclidean score),
//     10*6 -> 64 columns for n2: 288 bytes per row, the same
//     tile geometry as the Hamming engine (128 rows x 288 bytes, canonical K-major no-swizzle UMMA layout);
//   * hypothesis features depend on the camera of the correspondence (A = Rc^T R^T, b = -Rc^T (R^T t + tc)), so each
//     hypothesis tile exists once per camera, and each correspondence tile too (rows of the other camera are zero); a tile
//     that mixes cameras simply runs both MMAs into the same accumulator;
//   * an epilogue thread owns one hypothesis (= TMEM lane), reads 32 pairs of (s, n2) with tcgen05.ld and per pair does
//     one FFMA (s|s| + a constant of the hypothesis), one packed FFMA2 per two pairs for each of t = D - band and
//     u = D + band, and two SHF that collect their sign bits; 32 pairs are counted with one POPC.
// Exactness: a band bounds the error of D from the split, the accumulation and the two float32 operations:
// |err D| <= BAND_REL (|p|^2 + |b|^2).  Worst-case model (u = 2^-24; T = the sum of |terms| of an accumulator):
//   * float32 features: the hypothesis feature and the correspondence feature are each one rounding of a float64 value: 2u T;
//   * the split: the dropped products mid*lo, lo*mid, lo*lo are below 2^-24 + 2^-24 + 2^-32 of a term: 2u T;
//   * accumulation — the HARDWARE ASSUMPTION, not documented by NVIDIA: each tcgen05.mma kind::f16 instruction adds the exact
//     sum of its 16 products to the float32 accumulator and rounds once, to nearest (e = u) or toward zero (e = 2u); every
//     partial sum is at most T, so m instructions add m e T (m = 5 for s, 4 for n2).
//   So |err s| <= (4u + 5e) T_s and |err n2| <= (4u + 4e) T_n.  Bearing score (|f| = 1, A orthogonal, b of the pair's camera,
//   B = max_cam |b|, S = |p|^2 + B^2): T_s <= sqrt(3) |p| + |b|, |s| <= |p| + |b|, hence |err s|s|| <= 2|s| |err s| <=
//   6.2 S (4u + 5e); T_n <= (|p| + |b|)^2 + 1.52 B^2 <= 3.52 S; the epilogue adds the rounding of w (3.52 u S), of the constants
//   c^2 + BETA (2 x 3.52 u S) and of K_h against the shift inside N' (12.2 u S; the rounding of t itself cannot flip its sign).
//   Total 107 u S = 6.4e-6 S (0.49 BAND_REL) to nearest, 152 u S = 9.1e-6 S (0.70 BAND_REL) toward zero.
//   Measured through the PROBE instantiation on every pair of the test problems (tests/test_gpu_score_tc.py,
//   tests/test_gpu_score_stress.py: large motion, far points, points at the camera centre, s ~ 0 and s < 0, millimetres)
//   the error stays below a quarter of BAND_REL, which those tests assert.  Since x = A p + b with A orthogonal, |p|^2 <= 2 n2 + 2 |b|^2, so the
// band is at most BETA n2 + G_h with BETA = 2 BAND_REL and G_h = 3 BAND_REL |b_h|^2 = BETA * 1.5 |b_h|^2.  The constant of
// the hypothesis rides through the MMA: the n2 GEMM delivers N' = n2 + 1.5 |b_h|^2 (added to the hypothesis feature that
// multiplies the correspondence's constant 1), so the band is BETA N' and D = (s|s| + c^2 1.5 |b_h|^2) - c^2 N':
// t = w - (c^2 + BETA) N' >= 0 is a certain inlier, u = w - (c^2 - BETA) N' < 0 a certain outlier, with
// w = s|s| + K_h one FFMA.  The uncertain pairs of a chunk
// (bit mask) are queued and re-decided after the item by the scalar float32 path with ITS rigorous guard and, inside that,
// by inlier_exact() in float64 — the same deferred path score_kernel uses — so every count equals the float64 oracle's.
// Euclidean score (|A p + b - q| < thr, q = the current frame's 3D point): r^2 = s' + n2 with s' = |q|^2 - 2 q.(A p + b) — the
// same 13 hypothesis features against (-2 q_i p_k, -2 q_i, |q|^2) — and the same n2 GEMM, so both scores share tiles, MMA
// issue and pipeline; only the correspondence features and the epilogue arithmetic differ.  r^2 is a difference of large
// terms, so its band scales with |p|^2 + |q|^2 + |b|^2 =: S, not with r^2 (worst case, model above: T_s' <= 2 sqrt(3) |q||p| +
// 2 |q||b| + |q|^2 <= 3.73 S and T_n <= (|p| + |b|)^2 <= 2 S, so |err r^2| <= 49.6 u S = 3.0e-6 S (0.59 BAND_EUCLID) to nearest,
// 76.2 u S = 4.5e-6 S (0.91 BAND_EUCLID) toward zero; the epilogue's roundings scale with r^2 and thr^2, far inside the band's
// 2 B r^2 term; measured below a quarter of the band, as for the bearing score) — but both accumulators bound S: |p|^2 <= 2 n2 +
// 2 |b|^2 and, because r^2 = |q - x|^2 >= (|q| - |x|)^2, |q|^2 <= 2 n2 + 2 r^2.  So band <= B (4 n2 + 2 r^2 + 3 |b_h|^2) per
// pair: t = (thr^2 - 3B|b|^2) - (1 + 2B) r^2 - 4B n2 >= 0 is a certain inlier, u = (thr^2 + 3B|b|^2) - (1 - 2B) r^2 + 4B n2 < 0
// a certain outlier.
// (ransac.cu includes <cuda_bf16.h> and "tc_common.cuh" at file scope before this.)
#pragma once

namespace score_tc {
using namespace sos_tc;

constexpr int TILE = 128;
constexpr int KS = 13, KN = 10;                 // features of the first accumulator (s / s') and of n2
constexpr int ES = 80, EN = 64;                 // bf16 elements per row: 6 per feature, zero padded to a multiple of 16
constexpr int KB = (ES + EN) * 2;               // 288 bytes per row
constexpr int CHUNKS = KB / 16;                 // 18 core-matrix columns
constexpr int GROUP_BYTES = CHUNKS * 128;       // one 8-row group
constexpr int TILE_BYTES = (TILE / 8) * GROUP_BYTES;   // 36864
constexpr int STAGES = 3;
constexpr int EPI_WARPS = 16;                   // warps 0..15: epilogue, 4 per SM sub-partition
// The single-issue roles sit above the epilogue warps (measured equal to sitting below them: what slows them is sharing a
// scheduler with four busy epilogue warps at all — clock64 stamps: 780 cycles to issue four bulk copies, 890 cycles for a
// try_wait on an already completed barrier while the epilogue classifies).
// Two MMA-issuing warps (on different sub-partitions): one owns the s accumulator (5 instructions per tile and camera), the
// other the n2 accumulator (4) — the issue loop of a single warp, competing with four busy epilogue warps for issue slots,
// took ~1800 cycles per tile for 576 cycles of tensor work (ncu: stall_not_selected / dispatch on every instruction of it).
constexpr int W_PRODUCER = EPI_WARPS, W_MMA = EPI_WARPS + 1, W_MMA2 = EPI_WARPS + 2, W_ALLOC = EPI_WARPS + 3;
constexpr int THREADS = (EPI_WARPS + 4) * 32;
constexpr int ECAP = 1536;                      // chunks with uncertain pairs per work item held in shared memory (entry + bit mask)
constexpr int PCAP = 2048;                      // uncertain pairs expanded per round of the deferred pass
constexpr int SMEM_BYTES = (2 + STAGES) * TILE_BYTES + 256 + ECAP * 8 + PCAP * 4 + TILE * 4;
constexpr float PAD_N2 = 1e30f;                 // n2 feature of a padding correspondence: D = -c^2 1e30, a certain outlier
// |err D| <= BAND_REL (|p|^2 + max_cam |b|^2) (derivation at the top of this file: worst case 0.49 / 0.70 of it for rounding to
// nearest / toward zero per MMA instruction; the tests measure below a quarter of it and assert that)
constexpr float BAND_REL = 13.0f * 9.5367431640625e-07f + 5e-7f;
constexpr float BETA = 2.02f * BAND_REL;        // band <= BETA (n2 + B2_SHIFT |b|^2)
// Euclidean score: |err r^2| <= BAND_EUCLID (|p|^2 + |q|^2 + |b|^2) (worst case 0.59 / 0.91 of it; measured below a quarter)
constexpr float BAND_EUCLID = 5e-6f;
constexpr double B2_SHIFT = 1.52;               // (3 / 2 of the derivation, padded for the float32 rounding of |b|^2 in the epilogue)

struct TileMeta {
  uint32_t cam_mask;   // bit c: the tile holds correspondences of camera c
  float pq2;           // Euclidean score: max over the tile of |p|^2 + |q|^2 (the absolute part of its band)
};

// float32 -> three bfloat16 pieces with x == hi + mid + lo exactly
__device__ __forceinline__ void split3(float x, uint32_t& h, uint32_t& m, uint32_t& l) {
  const __nv_bfloat16 bh = __float2bfloat16_rn(x);
  const float r1 = x - __bfloat162float(bh);
  const __nv_bfloat16 bm = __float2bfloat16_rn(r1);
  const float r2 = r1 - __bfloat162float(bm);
  const __nv_bfloat16 bl = __float2bfloat16_rn(r2);
  h = __bfloat16_as_ushort(bh);
  m = __bfloat16_as_ushort(bm);
  l = __bfloat16_as_ushort(bl);
}

// One 288-byte row of a tile.  ROLE 0 (hypothesis, A operand): the six columns of a feature hold (h, h, m, h, l, m);
// ROLE 1 (correspondence, B operand): (h, m, h, l, h, m) — their products are hh + hm + mh + hl + lh + mm.
// Byte (row r, k) of a tile sits at (r / 8) * GROUP_BYTES + (k / 16) * 128 + (r % 8) * 16 + k % 16.
template <int ROLE>
__device__ __forceinline__ void write_row(uint8_t* __restrict__ tile, int r, const float* fs, const float* fn) {
  uint32_t e[(ES + EN) / 2];   // packed pairs of bf16
#pragma unroll
  for (int i = 0; i < (ES + EN) / 2; ++i) e[i] = 0u;
  auto put = [&](int base, int k, float x) {
    uint32_t h, m, l;
    split3(x, h, m, l);
    const uint32_t c0 = h, c1 = ROLE ? m : h, c2 = ROLE ? h : m, c3 = ROLE ? l : h, c4 = ROLE ? h : l, c5 = m;
    const int el = base + 6 * k;   // even
    e[el / 2 + 0] = c0 | (c1 << 16);
    e[el / 2 + 1] = c2 | (c3 << 16);
    e[el / 2 + 2] = c4 | (c5 << 16);
  };
#pragma unroll
  for (int k = 0; k < KS; ++k) put(0, k, fs[k]);
#pragma unroll
  for (int k = 0; k < KN; ++k) put(ES, k, fn[k]);
  uint8_t* row = tile + (size_t)(r >> 3) * GROUP_BYTES + (r & 7) * 16;
#pragma unroll
  for (int c = 0; c < CHUNKS; ++c)
    *(uint4*)(row + c * 128) = make_uint4(e[4 * c], e[4 * c + 1], e[4 * c + 2], e[4 * c + 3]);
}

// Hypothesis side, called by the hypothesize kernels: Ad (3x3 row-major) and bd of camera c in float64; bmax2 = the largest
// |b|^2 over the cameras of the rig (the band constant must not depend on the camera of the correspondence).
__device__ __forceinline__ void emit_hyp_row(uint8_t* __restrict__ tile, int r, const double* Ad, const double* bd, double bmax2,
                                             bool ok, int mode) {
  float fs[KS], fn[KN];
  if (ok) {
#pragma unroll
    for (int i = 0; i < 9; ++i) fs[i] = (float)Ad[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) fs[9 + i] = (float)bd[i];
    fs[12] = 1.f;   // against |q|^2 (Euclidean score; the bearing score's correspondence side holds 0 there)
    auto G = [&](int k, int l) { return Ad[k] * Ad[l] + Ad[3 + k] * Ad[3 + l] + Ad[6 + k] * Ad[6 + l]; };
    fn[0] = (float)G(0, 0); fn[1] = (float)G(1, 1); fn[2] = (float)G(2, 2);
    fn[3] = (float)G(0, 1); fn[4] = (float)G(0, 2); fn[5] = (float)G(1, 2);
#pragma unroll
    for (int k = 0; k < 3; ++k) fn[6 + k] = (float)(Ad[k] * bd[0] + Ad[3 + k] * bd[1] + Ad[6 + k] * bd[2]);
    // bearing score: N' = n2 + B2_SHIFT max |b|^2; Euclidean score: plain n2
    fn[9] = (float)(bd[0] * bd[0] + bd[1] * bd[1] + bd[2] * bd[2] + (mode == SOS_SCORE_BEARING ? B2_SHIFT * bmax2 : 0.0));
  } else {
    // failed model: NaN accumulators never land inside the band (no deferred work) and its count stays hugely negative
#pragma unroll
    for (int i = 0; i < KS; ++i) fs[i] = CUDART_NAN_F;
#pragma unroll
    for (int i = 0; i < KN; ++i) fn[i] = CUDART_NAN_F;
  }
  write_row<0>(tile, r, fs, fn);
}

// Correspondence side: one block per 128-row tile of one problem; both camera tiles are written (the other camera's row
// is zero), plus the tile's camera mask and max |p|^2.
__global__ void __launch_bounds__(TILE)
corr_expand_kernel(int mode, const float* __restrict__ p_ref, const float* __restrict__ f_cur, const uint8_t* __restrict__ cam,
                   const int32_t* __restrict__ n_arr, int cap, int n_cams, int ct, uint8_t* __restrict__ b_exp,
                   TileMeta* __restrict__ meta) {   // f_cur: bearings (bearing score) or the current frame's points (Euclidean)
  __shared__ float wmax[TILE / 32];
  const int b = blockIdx.y, tile = blockIdx.x, r = threadIdx.x;
  const int n = min(n_arr[b], cap);
  if (tile * TILE >= n) return;
  const int j = tile * TILE + r;
  float fs[KS], fn[KN];
#pragma unroll
  for (int i = 0; i < KS; ++i) fs[i] = 0.f;
#pragma unroll
  for (int i = 0; i < KN; ++i) fn[i] = 0.f;
  int c = 0;
  bool real = false;
  float pq2 = 0.f;
  if (j < n) {
    const size_t o = ((size_t)b * cap + j) * 3;
    const float p[3] = {p_ref[o], p_ref[o + 1], p_ref[o + 2]}, f[3] = {f_cur[o], f_cur[o + 1], f_cur[o + 2]};
    c = (n_cams > 1 && cam) ? (cam[(size_t)b * cap + j] ? 1 : 0) : 0;
    real = isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]) && isfinite(f[0]) && isfinite(f[1]) && isfinite(f[2]);
    if (real) {
#pragma unroll
      const double sc = mode == SOS_SCORE_BEARING ? 1.0 : -2.0;   // bearing: f_i p_k, f_i; Euclidean: -2 q_i p_k, -2 q_i, |q|^2
#pragma unroll
      for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int k = 0; k < 3; ++k) fs[i * 3 + k] = (float)(sc * (double)f[i] * (double)p[k]);
        fs[9 + i] = (float)(sc * (double)f[i]);
      }
      const double px = p[0], py = p[1], pz = p[2];
      if (mode != SOS_SCORE_BEARING) {
        const double q2 = (double)f[0] * f[0] + (double)f[1] * f[1] + (double)f[2] * f[2];
        fs[12] = (float)q2;
        pq2 = (float)(px * px + py * py + pz * pz + q2) * 1.000001f;
      }
      fn[0] = (float)(px * px); fn[1] = (float)(py * py); fn[2] = (float)(pz * pz);
      fn[3] = (float)(2.0 * px * py); fn[4] = (float)(2.0 * px * pz); fn[5] = (float)(2.0 * py * pz);
      fn[6] = 2.f * p[0]; fn[7] = 2.f * p[1]; fn[8] = 2.f * p[2];
      fn[9] = 1.f;
    }
  }
  // which cameras the tile holds (the MMA kernel never reads the tile of an absent camera, so it is not written either)
  const uint32_t mask = (uint32_t)__syncthreads_or((j < n && c == 0) ? 1 : 0) | ((uint32_t)__syncthreads_or((j < n && c == 1) ? 1 : 0) << 1);
  uint8_t* t0 = b_exp + ((size_t)((size_t)b * ct + tile) * 2) * TILE_BYTES;
  float zs[KS], zn[KN];
#pragma unroll
  for (int i = 0; i < KS; ++i) zs[i] = 0.f;
#pragma unroll
  for (int i = 0; i < KN; ++i) zn[i] = 0.f;
  if (!real) {
    // padding row, or a correspondence with a non-finite coordinate (NaN never passes the reference's test): n2 = 1e30 in
    // whichever camera tiles are multiplied
    fn[0] = PAD_N2;
    zn[0] = PAD_N2;
  }
  write_row<1>(t0 + (size_t)c * TILE_BYTES, r, fs, fn);
  if ((mask >> (c ^ 1)) & 1u) write_row<1>(t0 + (size_t)(c ^ 1) * TILE_BYTES, r, zs, zn);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) pq2 = fmaxf(pq2, __shfl_xor_sync(0xFFFFFFFFu, pq2, off));
  if ((r & 31) == 0) wmax[r >> 5] = pq2;
  __syncthreads();
  if (r == 0) {
    TileMeta m;
    m.cam_mask = mask;
    m.pq2 = fmaxf(fmaxf(wmax[0], wmax[1]), fmaxf(wmax[2], wmax[3]));
    meta[(size_t)b * ct + tile] = m;
  }
}

// instruction descriptor: D = F32 (1 << 4), A = B = BF16 (1 << 7, 1 << 10), both K-major, N = 128, M = 128
constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TILE >> 3) << 17) | ((uint32_t)(TILE >> 4) << 24);

struct Args {
  const uint8_t *a_exp, *b_exp;
  const TileMeta* meta;
  const int32_t* n_arr;
  int cap, n_hyp, ht, ct, splits;
  const HypRec* recs;
  int32_t* counts;
  const float *p_ref, *f_cur;   // f_cur: bearings, or the current frame's points (Euclidean score)
  const uint8_t* cam;
  ScoreConst k;
  float* probe;          // PROBE (may be NULL): (s, N') of every pair, [problem][hypothesis][ct * 128][2]
  int32_t* stats;        // PROBE (may be NULL): deferred-path counters, SOS_SCORE_STATS layout (include/sosfront.h)
};

// one deferred pair, decided exactly like score_kernel's deferred pass
template <int MODE>
__device__ __forceinline__ int exact_pair(const Args& a, const Rig& rig, int b, int h, int j, int n) {
  if (j >= n) return 0;
  const HypRec* hr = a.recs + (size_t)b * a.n_hyp + h;
  const size_t o = ((size_t)b * a.cap + j) * 3;
  const int c = (rig.n_cams > 1 && a.cam) ? (a.cam[(size_t)b * a.cap + j] ? 1 : 0) : 0;
  const float4 p = make_float4(a.p_ref[o], a.p_ref[o + 1], a.p_ref[o + 2], 0.f);
  const float4 q = make_float4(a.f_cur[o], a.f_cur[o + 1], a.f_cur[o + 2], 0.f);
  float Ax[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) Ax[i] = __ldg(&hr->xf[c][i]);
  float D, g;
  decision<MODE>(Ax, p, q, guard_of(MODE, p.x, p.y, p.z, q.x, q.y, q.z, a.k.thr), a.k, D, g);
  if (fabsf(D) < g) return inlier_exact(MODE, hr->pose64, rig, c, p, q, a.k.thr) ? 1 : 0;
  return D > 0.f ? 1 : 0;
}

__device__ __forceinline__ float2 pk_ffma2(float2 x, float2 y, float2 z) {
  float2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(reinterpret_cast<uint64_t&>(d))
      : "l"(reinterpret_cast<uint64_t&>(x)), "l"(reinterpret_cast<uint64_t&>(y)), "l"(reinterpret_cast<uint64_t&>(z)));
  return d;
}

// Work item = (problem, 128 hypotheses, a range of correspondence tiles); one CTA per item, warp-specialised like the
// Hamming engine: the producer warp streams the two hypothesis tiles (one per camera) and a ring of correspondence tiles
// with cp.async.bulk, one lane of the MMA warp issues 5 + 4 tcgen05.mma (M128 N128 K16) per (tile, camera) into a double-buffered
// accumulator pair (s: 128 columns, n2: 128 columns; 2 buffers = all 512 TMEM columns), warps 0..15 are the epilogue:
// warp group g takes the 32-pair chunk g of every tile.
template <bool PROBE, int MODE>
__global__ void __launch_bounds__(THREADS, 1) score_mma_kernel(const Args a, const __grid_constant__ Rig rig) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int item = blockIdx.x;
  const int b = item / (a.ht * a.splits), ht = (item / a.splits) % a.ht, split = item % a.splits;
  const int n = min(a.n_arr[b], a.cap);
  const int nt = (n + TILE - 1) / TILE;
  const int per = (nt + a.splits - 1) / a.splits;
  const int k_begin = min(nt, split * per), k_end = min(nt, k_begin + per);
  if (k_begin >= k_end) return;
  uint8_t* sA = smem;
  uint8_t* sB = smem + 2 * TILE_BYTES;
  uint64_t* bars = (uint64_t*)(smem + (2 + STAGES) * TILE_BYTES);
  constexpr int FULL = 0, EMPTY = STAGES, TFULL = 2 * STAGES, TEMPTY = 2 * STAGES + 2, AFULL = 2 * STAGES + 4;
  uint32_t* tmem_slot = (uint32_t*)(bars + AFULL + 1);
  int* q_n = (int*)(tmem_slot + 1);       // chunks queued
  int* p_n = q_n + 1;                     // pairs expanded in this round
  uint32_t* qent = (uint32_t*)(smem + (2 + STAGES) * TILE_BYTES + 256);   // tile << 9 | chunk << 7 | row
  uint32_t* qmask = qent + ECAP;                                           // uncertain pairs of the chunk (bit 31 - i = pair i)
  uint32_t* pairs = qmask + ECAP;                                          // entry << 5 | pair
  int* fixcnt = (int*)(pairs + PCAP);                                      // inliers found by the deferred pass, per hypothesis row
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  const TileMeta* meta = a.meta + (size_t)b * a.ct;

  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(BAR(FULL + i), 1); mbar_init(BAR(EMPTY + i), 2); }   // EMPTY, TFULL: one commit per MMA warp
    mbar_init(BAR(TFULL), 2); mbar_init(BAR(TFULL + 1), 2);
    mbar_init(BAR(TEMPTY), EPI_WARPS); mbar_init(BAR(TEMPTY + 1), EPI_WARPS);
    mbar_init(BAR(AFULL), 1);
    *q_n = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < TILE) fixcnt[tid] = 0;
  if (warp == W_ALLOC) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == W_PRODUCER) {
    // producer: the whole warp walks the tiles (camera masks prefetched one tile ahead: a dependent global load per tile in
    // this loop held the ring back), the elected lane issues the copies
    const uint8_t* ga = a.a_exp + ((size_t)((size_t)b * a.ht + ht) * 2) * TILE_BYTES;
    if (elect_one()) {
      mbar_expect_tx(BAR(AFULL), 2u * TILE_BYTES);
#pragma unroll
      for (int p = 0; p < 8; ++p) bulk_g2s(smem_u32(sA) + p * (TILE_BYTES / 4), ga + (size_t)p * (TILE_BYTES / 4), TILE_BYTES / 4, BAR(AFULL));
    }
    uint32_t t = 0;
    uint32_t mask = meta[k_begin].cam_mask;
    for (int k = k_begin; k < k_end; ++k) {
      const uint32_t mask_next = meta[min(k + 1, k_end - 1)].cam_mask;
      for (int c = 0; c < 2; ++c) {
        if (!((mask >> c) & 1u)) continue;
        const uint32_t s = t % STAGES;
        mbar_wait(BAR(EMPTY + s), ((t / STAGES) & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(BAR(FULL + s), TILE_BYTES);
          const uint8_t* gb = a.b_exp + ((size_t)(((size_t)b * a.ct + k) * 2 + c)) * TILE_BYTES;
          const uint32_t dst = smem_u32(sB) + s * TILE_BYTES;
#pragma unroll
          for (int p = 0; p < 4; ++p) bulk_g2s(dst + p * (TILE_BYTES / 4), gb + (size_t)p * (TILE_BYTES / 4), TILE_BYTES / 4, BAR(FULL + s));
        }
        __syncwarp();
        ++t;
      }
      mask = mask_next;
    }
  } else if (warp == W_MMA || warp == W_MMA2) {
    // MMA issuers: converged warps, elected lane (see elect_one); W_MMA owns the s accumulator, W_MMA2 the n2 accumulator
    const bool part_n = warp == W_MMA2;
    mbar_wait(BAR(AFULL), 0);
    uint32_t t = 0, it = 0;
    uint32_t mask = meta[k_begin].cam_mask;
    for (int k = k_begin; k < k_end; ++k, ++it) {
      const uint32_t mask_next = meta[min(k + 1, k_end - 1)].cam_mask;
      const uint32_t buf = it & 1;
      mbar_wait(BAR(TEMPTY + buf), ((it >> 1) & 1) ^ 1);   // the epilogue has drained this accumulator pair
      uint32_t acc = 0;
      for (int c = 0; c < 2; ++c) {
        if (!((mask >> c) & 1u)) continue;
        const uint32_t s = t % STAGES;
        mbar_wait(BAR(FULL + s), (t / STAGES) & 1);
        tc_fence_after();
        const uint64_t da = smem_desc(smem_u32(sA) + c * TILE_BYTES, GROUP_BYTES);
        const uint64_t db = smem_desc(smem_u32(sB) + s * TILE_BYTES, GROUP_BYTES);
        if (elect_one()) {
          if (!part_n) {
#pragma unroll
            for (int kk = 0; kk < ES / 16; ++kk)
              tc_mma<KIND_L2>(tmem + buf * 256, da + (uint64_t)(16 * kk), db + (uint64_t)(16 * kk), IDESC, acc | (kk > 0));
          } else {
#pragma unroll
            for (int kk = ES / 16; kk < (ES + EN) / 16; ++kk)
              tc_mma<KIND_L2>(tmem + buf * 256 + TILE, da + (uint64_t)(16 * kk), db + (uint64_t)(16 * kk), IDESC, acc | (kk > ES / 16));
          }
          tc_commit(BAR(EMPTY + s));
        }
        __syncwarp();
        acc = 1;
        ++t;
      }
      if (elect_one()) tc_commit(BAR(TFULL + buf));
      __syncwarp();
      mask = mask_next;
    }
  } else if (warp < EPI_WARPS) {
    const int g = warp >> 2, quarter = warp & 3;   // a warp may only touch the TMEM lanes of its quarter
    const int row = quarter * 32 + lane;
    const int h = ht * TILE + row;
    const bool valid_h = h < a.n_hyp;
    float bmax2 = 0.f;
    if (valid_h) {
      const HypRec* hr = a.recs + (size_t)b * a.n_hyp + h;
      for (int c = 0; c < rig.n_cams; ++c) {
        const float bx = __ldg(&hr->xf[c][9]), by = __ldg(&hr->xf[c][10]), bz = __ldg(&hr->xf[c][11]);
        bmax2 = fmaxf(bmax2, bx * bx + by * by + bz * bz);
      }
    }
    // Euclidean score: t = t_lo - e_lo r^2 - e_n n2,  u = t_hi - e_hi r^2 + e_n n2  (band = B (4 n2 + 2 r^2 + 3 |b|^2), padded 1 %)
    constexpr float EB = 1.01f * BAND_EUCLID;
    const float2 t_lo = make_float2(a.k.thr_sq - 3.f * EB * bmax2, a.k.thr_sq - 3.f * EB * bmax2);
    const float2 t_hi = make_float2(a.k.thr_sq + 3.f * EB * bmax2, a.k.thr_sq + 3.f * EB * bmax2);
    const float2 e_lo = make_float2(-(1.f + 2.f * EB), -(1.f + 2.f * EB)), e_hi = make_float2(-(1.f - 2.f * EB), -(1.f - 2.f * EB));
    const float2 e_np = make_float2(4.f * EB, 4.f * EB), e_nm = make_float2(-4.f * EB, -4.f * EB);
    const float Kh = a.k.cos_min_sq * (float)B2_SHIFT * bmax2;   // D = (s|s| + Kh) - c^2 N'
    const float2 ka = make_float2(-(a.k.cos_min_sq + BETA), -(a.k.cos_min_sq + BETA));
    const float2 kb = make_float2(-(a.k.cos_min_sq - BETA), -(a.k.cos_min_sq - BETA));
    int cnt = 0;
    uint32_t it = 0;
    for (int k = k_begin; k < k_end; ++k, ++it) {
      const uint32_t buf = it & 1;
      mbar_wait(BAR(TFULL + buf), (it >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem + ((uint32_t)(quarter * 32) << 16) + buf * 256 + g * 32;
      int sv[32], nv[32];
      tmem_ld32(taddr, sv);
      tmem_ld32(taddr + TILE, nv);
      tmem_ld_wait(sv);
      tmem_ld_wait(nv);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(TEMPTY + buf));     // this warp's share of the accumulator pair is in registers
      auto classify = [&](const int (&S)[32], const int (&N)[32], int chunk) {
        uint32_t mt = 0, mu = 0;       // sign bits of t and u: pair i ends up in bit 31 - i
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const float s0 = __int_as_float(S[i]), s1 = __int_as_float(S[i + 1]);
          const float2 n2 = make_float2(__int_as_float(N[i]), __int_as_float(N[i + 1]));
          float2 t, u;
          if (MODE == SOS_SCORE_BEARING) {
            // s|s| folds the s > 0 test into D
            const float2 w = make_float2(__fmaf_rn(s0, fabsf(s0), Kh), __fmaf_rn(s1, fabsf(s1), Kh));
            t = pk_ffma2(n2, ka, w);
            u = pk_ffma2(n2, kb, w);
          } else {
            // r^2 = s' + n2;  t >= 0: certain inlier,  u < 0: certain outlier (constants above)
            const float2 r2 = make_float2(__fadd_rn(s0, n2.x), __fadd_rn(s1, n2.y));
            t = pk_ffma2(n2, e_nm, pk_ffma2(r2, e_lo, t_lo));
            u = pk_ffma2(n2, e_np, pk_ffma2(r2, e_hi, t_hi));
          }
          mt = __funnelshift_l(__float_as_uint(t.x), mt, 1);
          mt = __funnelshift_l(__float_as_uint(t.y), mt, 1);
          mu = __funnelshift_l(__float_as_uint(u.x), mu, 1);
          mu = __funnelshift_l(__float_as_uint(u.y), mu, 1);
          if (PROBE && valid_h && a.probe) {
            float* o = a.probe + (((size_t)b * a.n_hyp + h) * ((size_t)a.ct * TILE) + (size_t)k * TILE + chunk * 32 + i) * 2;
            o[0] = s0; o[1] = n2.x; o[2] = s1; o[3] = n2.y;
          }
        }
        if (!valid_h) return;
        const uint32_t unsure = mt & ~mu;          // t < 0 <= u
        cnt += 32 - __popc(mt);                    // certain inliers; uncertain pairs are added by the deferred pass
        if (unsure) {
          const int slot = atomicAdd(q_n, 1);
          if (slot < ECAP) {
            qent[slot] = ((uint32_t)k << 9) | ((uint32_t)chunk << 7) | (uint32_t)row;
            qmask[slot] = unsure;
          } else {   // queue full (far-field Euclidean batches): this thread decides its uncertain pairs on its own
            for (int i = 0; i < 32; ++i)
              if ((unsure >> (31 - i)) & 1u) cnt += exact_pair<MODE>(a, rig, b, h, k * TILE + chunk * 32 + i, n);
          }
        }
      };
      classify(sv, nv, g);
    }
    // deferred pass over the uncertain pairs, all 256 epilogue threads: expand the chunk masks into a pair list (in rounds
    // of PCAP pairs), one thread per pair
    const int te = tid;
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
    const int nq = min(*q_n, ECAP);
    int rounds = 0, expanded = 0;   // PROBE statistics
    for (bool more = nq > 0; more;) {
      if (te == 0) *p_n = 0;
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
      for (int e = te; e < nq; e += EPI_WARPS * 32) {
        uint32_t m = qmask[e];
        while (m) {
          const int slot = atomicAdd(p_n, 1);
          if (slot >= PCAP) break;
          const int bit = 31 - __clz(m);
          pairs[slot] = ((uint32_t)e << 5) | (uint32_t)(31 - bit);
          m &= ~(1u << bit);
        }
        qmask[e] = m;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
      const int np = *p_n;
      for (int x = te; x < min(np, PCAP); x += EPI_WARPS * 32) {
        const uint32_t v = pairs[x], ent = qent[v >> 5];
        const int k = (int)(ent >> 9), chunk = (int)((ent >> 7) & 3u), r = (int)(ent & 127u);
        if (exact_pair<MODE>(a, rig, b, ht * TILE + r, k * TILE + chunk * 32 + (int)(v & 31u), n)) atomicAdd(&fixcnt[r], 1);
      }
      more = np > PCAP;
      ++rounds;
      expanded += min(np, PCAP);
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
    }
    if (PROBE && a.stats && te == 0) {
      const int queued = *q_n;
      atomicAdd(&a.stats[SOS_STAT_TC_ITEMS], 1);
      atomicAdd(&a.stats[SOS_STAT_TC_CHUNKS], queued);
      atomicMax(&a.stats[SOS_STAT_TC_CHUNKS_MAX], queued);
      atomicAdd(&a.stats[SOS_STAT_TC_CHUNKS_IN_THREAD], max(queued - ECAP, 0));
      atomicAdd(&a.stats[SOS_STAT_TC_PAIRS], expanded);
      atomicMax(&a.stats[SOS_STAT_TC_ROUNDS_MAX], rounds);
    }
    if (g == 0) cnt += fixcnt[row];
    if (valid_h && cnt != 0) atomicAdd(&a.counts[(size_t)b * a.n_hyp + h], cnt);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == W_ALLOC) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}

inline size_t scratch_bytes(int n_problems, int n_hyp, int cap) {
  const size_t ht = (size_t)(n_hyp + TILE - 1) / TILE, ct = (size_t)(cap + TILE - 1) / TILE;
  return (size_t)n_problems * (ht + ct) * 2 * TILE_BYTES + sos_align_up((size_t)n_problems * ct * sizeof(TileMeta), 256) + 512;
}

}  // namespace score_tc
