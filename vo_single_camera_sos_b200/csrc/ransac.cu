// Step 5 of the SOS front-end: batched RANSAC for rigid 3D-3D registration.
//
// Hypotheses are Arun/Kabsch fits on 3 correspondences, restating transformations.superimposition_matrix(v0, v1,
// scale=False, usesvd=True) (reference omnistereo/transformations.py:874-1030); the inlier score is either the
// Euclidean residual or the bearing-angle score of get_selected_distances_to_model (pose_est_tools.py:150-203, with
// the non-central correction of its comment at :181-185), i.e. what OpenGV's AbsolutePoseSacProblem evaluates.
//
// Four kernels per call, all on one stream:
//   hypothesize  one thread per (problem, hypothesis): sample rows, 3-point Kabsch in float64 (Jacobi on H^T H),
//                emit [R|t] and, per camera, the scoring transform  x = A p_ref + b  with A = Rc^T R^T,
//                b = -Rc^T (R^T t + tc)   (float32);
//   score        FP32-FMA bound: a thread keeps RS_HPT hypotheses (A, b) in registers and walks the block's chunk of
//                correspondences staged in shared memory (every lane reads the SAME point: broadcast LDS.128);
//                per pair 9 FMA (x) + 3 ADD + 3 FMA (|x - p_cur|^2) + compare; counts go to global with one
//                atomicAdd per (hypothesis, chunk);
//   argmax       one block per problem: packed key (count+1) << 32 | (0xFFFFFFFF - global hypothesis index), so
//                max() prefers the lowest index on ties (and reduces across GPUs with a plain 64-bit MAX);
//   mask         re-evaluates the winner with the very same float32 instruction sequence -> inlier mask.
#include <math_constants.h>
#include <stddef.h>

#include <cuda_bf16.h>

#include "sos_common.cuh"
#include "tc_common.cuh"

namespace {

// ------------------------------------------------------------------------------------------------------------
// float64 3x3 helpers (row-major)
// ------------------------------------------------------------------------------------------------------------
// Rotation R (det +1) maximising trace(R^T ... ) for covariance Hm = sum v1_i v0_i^T, i.e. U diag(1,1,det(U V^T)) V^T of
// Hm = U S V^T (transformations.py:942-953).  Returns false when the second singular value vanishes (rank < 2).
// V comes from one-sided (Hestenes) Jacobi on the columns of Hm, not from the eigenvectors of Hm^T Hm: forming Hm^T Hm squares
// the ratio of the singular values, so for a thin sample triangle (sigma2 / sigma1 ~ 1e-2) the second singular vector, and
// with it the pose, lost six digits against the float64 SVD of the oracle and inlier counts differed from it.
__device__ bool kabsch_rotation(const double* Hm, double* R) {
  double A[9], V[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
#pragma unroll
  for (int i = 0; i < 9; ++i) A[i] = Hm[i];
  for (int sweep = 0; sweep < 30; ++sweep) {
    bool rotated = false;
#pragma unroll
    for (int pq = 0; pq < 3; ++pq) {
      const int p = pq == 2 ? 1 : 0, q = pq == 0 ? 1 : 2;
      double alpha = 0.0, beta = 0.0, gamma = 0.0;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        alpha += A[k * 3 + p] * A[k * 3 + p];
        beta += A[k * 3 + q] * A[k * 3 + q];
        gamma += A[k * 3 + p] * A[k * 3 + q];
      }
      if (!(fabs(gamma) > 1e-15 * sqrt(alpha * beta))) continue;   // columns orthogonal to working precision
      rotated = true;
      const double zeta = (beta - alpha) / (2.0 * gamma);
      const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
      const double c = 1.0 / sqrt(1.0 + t * t), s = t * c;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const double ap = A[k * 3 + p], aq = A[k * 3 + q];
        A[k * 3 + p] = c * ap - s * aq;
        A[k * 3 + q] = s * ap + c * aq;
        const double vp = V[k * 3 + p], vq = V[k * 3 + q];
        V[k * 3 + p] = c * vp - s * vq;
        V[k * 3 + q] = s * vp + c * vq;
      }
    }
    if (!rotated) break;
  }
  // pick the two largest singular values (squared: the column norms of Hm V)
  double lam[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) lam[j] = A[j] * A[j] + A[3 + j] * A[3 + j] + A[6 + j] * A[6 + j];
  int i0 = 0;
  if (lam[1] > lam[i0]) i0 = 1;
  if (lam[2] > lam[i0]) i0 = 2;
  int i1 = (i0 + 1) % 3, i2 = (i0 + 2) % 3;
  if (lam[i2] > lam[i1]) { const int tmp = i1; i1 = i2; i2 = tmp; }
  if (!(lam[i0] > 0.0) || !(lam[i1] > 1e-24 * lam[i0])) return false;
  double v1[3] = {V[0 * 3 + i0], V[1 * 3 + i0], V[2 * 3 + i0]};
  double v2[3] = {V[0 * 3 + i1], V[1 * 3 + i1], V[2 * 3 + i1]};
  double u1[3], u2[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    u1[i] = Hm[i * 3 + 0] * v1[0] + Hm[i * 3 + 1] * v1[1] + Hm[i * 3 + 2] * v1[2];
    u2[i] = Hm[i * 3 + 0] * v2[0] + Hm[i * 3 + 1] * v2[1] + Hm[i * 3 + 2] * v2[2];
  }
  double n1 = sqrt(u1[0] * u1[0] + u1[1] * u1[1] + u1[2] * u1[2]);
  if (!(n1 > 0.0)) return false;
#pragma unroll
  for (int i = 0; i < 3; ++i) u1[i] /= n1;
  const double d12 = u1[0] * u2[0] + u1[1] * u2[1] + u1[2] * u2[2];
#pragma unroll
  for (int i = 0; i < 3; ++i) u2[i] -= d12 * u1[i];
  double n2 = sqrt(u2[0] * u2[0] + u2[1] * u2[1] + u2[2] * u2[2]);
  if (!(n2 > 0.0)) return false;
#pragma unroll
  for (int i = 0; i < 3; ++i) u2[i] /= n2;
  const double u3[3] = {u1[1] * u2[2] - u1[2] * u2[1], u1[2] * u2[0] - u1[0] * u2[2], u1[0] * u2[1] - u1[1] * u2[0]};
  const double v3[3] = {v1[1] * v2[2] - v1[2] * v2[1], v1[2] * v2[0] - v1[0] * v2[2], v1[0] * v2[1] - v1[1] * v2[0]};
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) R[i * 3 + j] = u1[i] * v1[j] + u2[i] * v2[j] + u3[i] * v3[j];
  return true;
}

// Arun on k points held in local arrays (v0 -> v1): M = [R|t] row-major 3x4 with v1 ~ R v0 + t.
__device__ bool arun_fit(const double* v0, const double* v1, int k, double* M) {
  double c0[3] = {0, 0, 0}, c1[3] = {0, 0, 0};
  for (int i = 0; i < k; ++i)
#pragma unroll
    for (int d = 0; d < 3; ++d) { c0[d] += v0[3 * i + d]; c1[d] += v1[3 * i + d]; }
#pragma unroll
  for (int d = 0; d < 3; ++d) { c0[d] /= (double)k; c1[d] /= (double)k; }
  double Hm[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = 0; i < k; ++i) {
    const double a[3] = {v0[3 * i] - c0[0], v0[3 * i + 1] - c0[1], v0[3 * i + 2] - c0[2]};
    const double b[3] = {v1[3 * i] - c1[0], v1[3 * i + 1] - c1[1], v1[3 * i + 2] - c1[2]};
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) Hm[r * 3 + c] += b[r] * a[c];  // dot(v1, v0.T), transformations.py:944
  }
  double R[9];
  if (!kabsch_rotation(Hm, R)) return false;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    M[r * 4 + 0] = R[r * 3 + 0]; M[r * 4 + 1] = R[r * 3 + 1]; M[r * 4 + 2] = R[r * 3 + 2];
    M[r * 4 + 3] = c1[r] - (R[r * 3 + 0] * c0[0] + R[r * 3 + 1] * c0[1] + R[r * 3 + 2] * c0[2]);
  }
  return true;
}

// sin^2 of the angle at vertex 0 of a triangle; collinear / coincident samples give ~0
__device__ __forceinline__ bool triangle_degenerate(const double* p) {
  const double e1[3] = {p[3] - p[0], p[4] - p[1], p[5] - p[2]}, e2[3] = {p[6] - p[0], p[7] - p[1], p[8] - p[2]};
  const double cx = e1[1] * e2[2] - e1[2] * e2[1], cy = e1[2] * e2[0] - e1[0] * e2[2], cz = e1[0] * e2[1] - e1[1] * e2[0];
  const double a2 = cx * cx + cy * cy + cz * cz;
  const double l1 = e1[0] * e1[0] + e1[1] * e1[1] + e1[2] * e1[2], l2 = e2[0] * e2[0] + e2[1] * e2[1] + e2[2] * e2[2];
  return !(a2 > 1e-12 * l1 * l2);
}

// ------------------------------------------------------------------------------------------------------------
// Per-hypothesis record in the scratch arena
// ------------------------------------------------------------------------------------------------------------
constexpr int RS_MAX_CAMS = 2;
struct Rig {
  double Rt[RS_MAX_CAMS][12];  // per camera row-major [Rc|tc]
  int n_cams;
};

struct HypRec {
  double pose64[12];              // [R|t] in float64: the exact (slow) path of the inlier test
  float pose[12];                 // [R|t], p_ref ~ R p_cur + t
  float xf[RS_MAX_CAMS][12];      // per camera: A (9, row-major) then b (3):  x = A p_ref + b
};

// ------------------------------------------------------------------------------------------------------------
// The inlier test.
//
// Fast path: float32 FMAs on the per-hypothesis transform.  It also produces a rigorous bound `guard` on its own
// rounding error; when the decision variable D lies inside the guard band the pair is re-evaluated by
// inlier_exact() in float64 with the reference's own formula.  The decision therefore equals the float64 decision
// (up to ~1e-15 relative), which is what makes inlier SETS bit-exact against the NumPy oracle, while >99.9 % of the
// pairs never leave the FP32 pipe.
//
// Error model (p, q are exact float32 inputs, A and b are float32 roundings of float64 values, u = 2^-24):
//   each component of x = A p + b:   |err| <= E = 4u (|p|_1 + |b|_inf),  and  |b|_inf <= |x|_2 + |p|_2
//   EUCLID : D = |x - q|^2 - thr^2;  within the band |x|_2 <= |q|_2 + 2 thr, |x - q|_1 <= 2 sqrt(3) thr, hence
//            |err D| <= u (28 thr (2|p|_1 + |q|_1 + 2 thr) + 18 thr^2) =: guard_j   (per correspondence, staged in .w)
//   BEARING: D = s^2 - c^2 |x|^2, s = f.x, c = 1 - thr;  |err D| <= u (80 |x|^2 + 32 |p|_1^2) = k |x|^2 + guard_j
// ------------------------------------------------------------------------------------------------------------
struct ScoreConst {
  float thr_sq;       // EUCLID: thr^2
  float cos_min_sq;   // BEARING: (1 - thr)^2
  float guard_rel;    // BEARING: 80 u
  double thr;         // the threshold itself, for the exact path
};

__device__ __noinline__ bool inlier_exact(int mode, const double* __restrict__ M, const Rig& rig, int cam, float4 p,
                                          float4 q, double thr) {
  const double px = p.x, py = p.y, pz = p.z;
  if (mode == SOS_SCORE_EUCLID) {
    // |p_ref - (R p_cur + t)| < thr
    const double cx = q.x, cy = q.y, cz = q.z;
    const double dx = px - (M[0] * cx + M[1] * cy + M[2] * cz + M[3]);
    const double dy = py - (M[4] * cx + M[5] * cy + M[6] * cz + M[7]);
    const double dz = pz - (M[8] * cx + M[9] * cy + M[10] * cz + M[11]);
    return sqrt(dx * dx + dy * dy + dz * dz) < thr;
  }
  // 1 - f . normalize(Rc^T (R^T (p - t) - tc)) < thr   (pose_est_tools.py:150-203, 181-185)
  const double ex = px - M[3], ey = py - M[7], ez = pz - M[11];
  double bx = M[0] * ex + M[4] * ey + M[8] * ez;
  double by = M[1] * ex + M[5] * ey + M[9] * ez;
  double bz = M[2] * ex + M[6] * ey + M[10] * ez;
  const double* C = rig.Rt[cam];
  bx -= C[3]; by -= C[7]; bz -= C[11];
  const double x = C[0] * bx + C[4] * by + C[8] * bz;
  const double y = C[1] * bx + C[5] * by + C[9] * bz;
  const double z = C[2] * bx + C[6] * by + C[10] * bz;
  const double nrm = sqrt(x * x + y * y + z * z);
  return 1.0 - ((double)q.x * (x / nrm) + (double)q.y * (y / nrm) + (double)q.z * (z / nrm)) < thr;
}

// Returns the fast decision in `in` and whether it is uncertain.
// Decision variable D (inlier <=> D > 0) and the bound g of its float32 rounding error (uncertain <=> |D| < g).
template <int MODE>
__device__ __forceinline__ void decision(const float* __restrict__ A, const float4& p, const float4& q, float guard_j,
                                         const ScoreConst& k, float& D, float& g) {
  const float x = __fmaf_rn(A[2], p.z, __fmaf_rn(A[1], p.y, __fmaf_rn(A[0], p.x, A[9])));
  const float y = __fmaf_rn(A[5], p.z, __fmaf_rn(A[4], p.y, __fmaf_rn(A[3], p.x, A[10])));
  const float z = __fmaf_rn(A[8], p.z, __fmaf_rn(A[7], p.y, __fmaf_rn(A[6], p.x, A[11])));
  if (MODE == SOS_SCORE_EUCLID) {
    const float dx = __fsub_rn(x, q.x), dy = __fsub_rn(y, q.y), dz = __fsub_rn(z, q.z);
    const float r2 = __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
    D = __fsub_rn(k.thr_sq, r2);
    g = guard_j;
  } else {
    const float s = __fmaf_rn(q.z, z, __fmaf_rn(q.y, y, __fmul_rn(q.x, x)));
    const float n2 = __fmaf_rn(z, z, __fmaf_rn(y, y, __fmul_rn(x, x)));
    D = __fmaf_rn(s, fabsf(s), -__fmul_rn(k.cos_min_sq, n2));  // s|s| folds the s > 0 test into D
    g = __fmaf_rn(k.guard_rel, n2, guard_j);
  }
}

__device__ __forceinline__ float guard_of(int mode, float px, float py, float pz, float qx, float qy, float qz, double thr) {
  const double u = 5.9604644775390625e-08;  // 2^-24
  const double p1 = fabs((double)px) + fabs((double)py) + fabs((double)pz);
  if (mode == SOS_SCORE_EUCLID) {
    const double q1 = fabs((double)qx) + fabs((double)qy) + fabs((double)qz);
    return (float)(u * (28.0 * thr * (2.0 * p1 + q1 + 2.0 * thr) + 18.0 * thr * thr) * 1.0001);
  }
  return (float)(u * 32.0 * p1 * p1 * 1.0001);
}

#include "score_mma.cuh"

// `tc_tile` (may be NULL): the two per-camera hypothesis tiles of the tensor-core score engine this hypothesis belongs to
// (score_mma.cuh); row `tc_row` of each gets the float64-derived features of that camera's transform.
__device__ void make_scoring_transforms(const double* M, const Rig& rig, HypRec& rec, uint8_t* tc_tile, int tc_row, int tc_mode) {
#pragma unroll
  for (int i = 0; i < 12; ++i) {
    rec.pose64[i] = M[i];
    rec.pose[i] = (float)M[i];
  }
  // body frame: y = R^T (p - t)
  double Rt_[9], bt[3];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) Rt_[i * 3 + j] = M[j * 4 + i];
#pragma unroll
  for (int i = 0; i < 3; ++i) bt[i] = -(Rt_[i * 3] * M[3] + Rt_[i * 3 + 1] * M[7] + Rt_[i * 3 + 2] * M[11]);
  double Ad[RS_MAX_CAMS][9], bd[RS_MAX_CAMS][3], bmax2 = 0.0;
  for (int c = 0; c < RS_MAX_CAMS; ++c) {
    if (c >= rig.n_cams) {
#pragma unroll
      for (int i = 0; i < 12; ++i) rec.xf[c][i] = 0.f;
      continue;
    }
    const double* C = rig.Rt[c];  // x = Rc^T (y - tc)
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
      for (int j = 0; j < 3; ++j) Ad[c][i * 3 + j] = C[0 * 4 + i] * Rt_[0 * 3 + j] + C[1 * 4 + i] * Rt_[1 * 3 + j] + C[2 * 4 + i] * Rt_[2 * 3 + j];
      bd[c][i] = C[0 * 4 + i] * (bt[0] - C[3]) + C[1 * 4 + i] * (bt[1] - C[7]) + C[2 * 4 + i] * (bt[2] - C[11]);
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) rec.xf[c][i] = (float)Ad[c][i];
#pragma unroll
    for (int i = 0; i < 3; ++i) rec.xf[c][9 + i] = (float)bd[c][i];
    bmax2 = fmax(bmax2, bd[c][0] * bd[c][0] + bd[c][1] * bd[c][1] + bd[c][2] * bd[c][2]);
  }
  if (tc_tile)
    for (int c = 0; c < rig.n_cams; ++c) score_tc::emit_hyp_row(tc_tile + (size_t)c * score_tc::TILE_BYTES, tc_row, Ad[c], bd[c], bmax2, true, tc_mode);
}

// a failed model: NaN never passes the inlier test
__device__ void make_failed_model(const Rig& rig, HypRec& rec, uint8_t* tc_tile, int tc_row, int tc_mode) {
#pragma unroll
  for (int i = 0; i < 12; ++i) {
    rec.pose[i] = CUDART_NAN_F;
    rec.pose64[i] = CUDART_NAN;
  }
  for (int c = 0; c < RS_MAX_CAMS; ++c) {
#pragma unroll
    for (int i = 0; i < 12; ++i) rec.xf[c][i] = CUDART_NAN_F;
    if (tc_tile && c < rig.n_cams) score_tc::emit_hyp_row(tc_tile + (size_t)c * score_tc::TILE_BYTES, tc_row, nullptr, nullptr, 0.0, false, tc_mode);
  }
}

__global__ void __launch_bounds__(128)
hypothesize_kernel(const float* __restrict__ p_ref, const float* __restrict__ p_cur, const int32_t* __restrict__ n_arr,
                   int cap, const uint32_t* __restrict__ hyp, int hyp_stride_problem, int n_hyp, Rig rig,
                   HypRec* __restrict__ recs, int32_t* __restrict__ counts, uint8_t* __restrict__ tc_a, int tc_mode) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (h >= n_hyp) return;
  const int n = n_arr[b];
  const uint32_t* hr = hyp + (size_t)b * hyp_stride_problem + (size_t)h * 3;
  uint8_t* tc_tile = tc_a ? tc_a + ((size_t)b * gridDim.x + blockIdx.x) * 2 * score_tc::TILE_BYTES : nullptr;  // 128 threads = one tile
  bool ok = n >= 3;
  int rows[3] = {0, 0, 0};
  if (ok) {
#pragma unroll
    for (int j = 0; j < 3; ++j) rows[j] = (int)(((uint64_t)hr[j] * (uint64_t)n) >> 32);
    ok = rows[0] != rows[1] && rows[0] != rows[2] && rows[1] != rows[2];
  }
  double v0[9], v1[9], M[12];
  if (ok) {
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const size_t o = ((size_t)b * cap + rows[j]) * 3;
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        v0[3 * j + d] = (double)p_cur[o + d];
        v1[3 * j + d] = (double)p_ref[o + d];
      }
    }
    ok = !triangle_degenerate(v0) && !triangle_degenerate(v1);
  }
  if (ok) ok = arun_fit(v0, v1, 3, M);
  HypRec rec;
  if (ok) make_scoring_transforms(M, rig, rec, tc_tile, (int)threadIdx.x, tc_mode);
  else make_failed_model(rig, rec, tc_tile, (int)threadIdx.x, tc_mode);
  recs[(size_t)b * n_hyp + h] = rec;
  counts[(size_t)b * n_hyp + h] = ok ? 0 : -(1 << 30);  // failed model: stays negative whatever is added
}

// ------------------------------------------------------------------------------------------------------------
// Bearing-only hypotheses (what the reference hands to OpenGV, pose_est_tools.py:785, 915: bearings of the current frame and
// 3D points of the reference frame only).  Four sampled rows: three for the minimal problem, the fourth picks among its
// solutions (OpenGV's sample size for its three-point solvers).  Depths along the three rays from Grunert's three-point
// problem (common origin: quartic in v = s3/s1, solved by Ferrari's closed form and polished), then Newton on the three
// distance equations with every ray's own origin (non-central rig), pose from the two congruent triangles.
// ------------------------------------------------------------------------------------------------------------
constexpr int P3P_NEWTON_ITERS = 8;

__device__ __forceinline__ double poly4(const double* c, double x) { return (((c[4] * x + c[3]) * x + c[2]) * x + c[1]) * x + c[0]; }
__device__ __forceinline__ double dpoly4(const double* c, double x) { return ((4.0 * c[4] * x + 3.0 * c[3]) * x + 2.0 * c[2]) * x + c[1]; }

// largest real root of m^3 + A m^2 + B m + C
__device__ double cubic_largest_root(double A, double B, double C) {
  const double P = B - A * A / 3.0, Q = 2.0 * A * A * A / 27.0 - A * B / 3.0 + C;
  const double disc = 0.25 * Q * Q + P * P * P / 27.0;
  double z;
  if (disc > 0.0) {
    const double sd = sqrt(disc);
    z = cbrt(-0.5 * Q + sd) + cbrt(-0.5 * Q - sd);
  } else if (P < 0.0) {
    const double k = sqrt(-P / 3.0);
    double arg = -0.5 * Q / (k * k * k);
    arg = fmin(1.0, fmax(-1.0, arg));
    z = 2.0 * k * cos(acos(arg) / 3.0);
  } else {
    z = 0.0;
  }
  double m = z - A / 3.0;
  for (int it = 0; it < 2; ++it) {
    const double f = ((m + A) * m + B) * m + C, df = (3.0 * m + 2.0 * A) * m + B;
    if (df != 0.0) m -= f / df;
  }
  return m;
}

// real roots of c[4] x^4 + ... + c[0] (c[4] != 0), each polished on the quartic itself; returns their number
__device__ int quartic_real_roots(const double* c, double* x) {
  const double a = c[3] / c[4], b = c[2] / c[4], cc = c[1] / c[4], d = c[0] / c[4];
  const double a2 = a * a;
  const double p = b - 0.375 * a2;
  const double q = cc - 0.5 * a * b + 0.125 * a2 * a;
  const double r = d - 0.25 * a * cc + 0.0625 * a2 * b - (3.0 / 256.0) * a2 * a2;
  double y[4];
  int n = 0;
  const double m = cubic_largest_root(p, 0.25 * p * p - r, -0.125 * q * q);
  const double tiny = 1e-13 * fmax(1.0, fmax(fabs(p), sqrt(fabs(r))));
  if (m > tiny) {
    // y^4 + p y^2 + q y + r = (y^2 - s y + p/2 + m + q/(2s)) (y^2 + s y + p/2 + m - q/(2s)),  s = sqrt(2m)
    const double s = sqrt(2.0 * m), h = 0.5 * p + m, g = q / (2.0 * s);
#pragma unroll
    for (int sign = 0; sign < 2; ++sign) {
      const double lin = sign ? s : -s, con = sign ? h - g : h + g;
      double disc = lin * lin - 4.0 * con;
      if (disc < 0.0 && disc > -1e-12 * fmax(1.0, fmax(lin * lin, fabs(con)))) disc = 0.0;
      if (disc >= 0.0) {
        const double sd = sqrt(disc);
        y[n++] = 0.5 * (-lin + sd);
        y[n++] = 0.5 * (-lin - sd);
      }
    }
  } else {
    // biquadratic: y^2 = (-p +- sqrt(p^2 - 4r)) / 2
    double disc = p * p - 4.0 * r;
    if (disc < 0.0 && disc > -1e-12 * fmax(1.0, p * p)) disc = 0.0;
    if (disc >= 0.0) {
      const double sd = sqrt(disc);
#pragma unroll
      for (int sign = 0; sign < 2; ++sign) {
        const double y2 = 0.5 * (-p + (sign ? -sd : sd));
        if (y2 >= 0.0) {
          y[n++] = sqrt(y2);
          y[n++] = -sqrt(y2);
        }
      }
    }
  }
  for (int i = 0; i < n; ++i) {
    double v = y[i] - 0.25 * a;
    for (int it = 0; it < 2; ++it) {
      const double df = dpoly4(c, v);
      if (df != 0.0) v -= poly4(c, v) / df;
    }
    x[i] = v;
  }
  return n;
}

__device__ __forceinline__ void cross3(const double* a, const double* b, double* o) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ __forceinline__ double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

// orthonormal frame (columns e1, e2, e3 stored as rows of F) on the first two edges of a triangle T [3][3]
__device__ __forceinline__ void triangle_frame(const double* T, double* F) {
  double e1[3] = {T[3] - T[0], T[4] - T[1], T[5] - T[2]}, w[3] = {T[6] - T[0], T[7] - T[1], T[8] - T[2]}, e3[3], e2[3];
  const double n1 = 1.0 / sqrt(dot3(e1, e1));
  e1[0] *= n1; e1[1] *= n1; e1[2] *= n1;
  cross3(e1, w, e3);
  const double n3 = 1.0 / sqrt(dot3(e3, e3));
  e3[0] *= n3; e3[1] *= n3; e3[2] *= n3;
  cross3(e3, e1, e2);
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    F[d] = e1[d];
    F[3 + d] = e2[d];
    F[6 + d] = e3[d];
  }
}

__global__ void __launch_bounds__(128)
hypothesize_p3p_kernel(const float* __restrict__ p_ref, const float* __restrict__ f_cur, const uint8_t* __restrict__ cam,
                       const int32_t* __restrict__ n_arr, int cap, const uint32_t* __restrict__ hyp, int hyp_stride_problem,
                       int n_hyp, Rig rig, HypRec* __restrict__ recs, int32_t* __restrict__ counts, uint8_t* __restrict__ tc_a, int tc_mode) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (h >= n_hyp) return;
  const int n = n_arr[b];
  const uint32_t* hr = hyp + (size_t)b * hyp_stride_problem + (size_t)h * 4;
  uint8_t* tc_tile = tc_a ? tc_a + ((size_t)b * gridDim.x + blockIdx.x) * 2 * score_tc::TILE_BYTES : nullptr;
  bool ok = n >= 4;
  int rows[4] = {0, 0, 0, 0};
  if (ok) {
#pragma unroll
    for (int j = 0; j < 4; ++j) rows[j] = (int)(((uint64_t)hr[j] * (uint64_t)n) >> 32);
    ok = rows[0] != rows[1] && rows[0] != rows[2] && rows[1] != rows[2] && rows[3] != rows[0] && rows[3] != rows[1] &&
         rows[3] != rows[2];
  }
  double P[12], dir[9], org[9], f4[3];
  int cam4 = 0;
  if (ok) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const size_t o = ((size_t)b * cap + rows[j]);
      const int c = cam ? min((int)cam[o], rig.n_cams - 1) : 0;
      const double f[3] = {(double)f_cur[o * 3], (double)f_cur[o * 3 + 1], (double)f_cur[o * 3 + 2]};
#pragma unroll
      for (int d = 0; d < 3; ++d) P[3 * j + d] = (double)p_ref[o * 3 + d];
      if (j < 3) {
        const double* C = rig.Rt[c];
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          dir[3 * j + d] = C[4 * d] * f[0] + C[4 * d + 1] * f[1] + C[4 * d + 2] * f[2];
          org[3 * j + d] = C[4 * d + 3];
        }
      } else {
        cam4 = c;
        f4[0] = f[0]; f4[1] = f[1]; f4[2] = f[2];
      }
    }
    ok = !triangle_degenerate(P);
  }
  double best_M[12];
  double best_res = CUDART_INF;
  if (ok) {
    double e[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) e[d] = P[3 + d] - P[6 + d];
    const double a2 = dot3(e, e);
#pragma unroll
    for (int d = 0; d < 3; ++d) e[d] = P[d] - P[6 + d];
    const double b2 = dot3(e, e);
#pragma unroll
    for (int d = 0; d < 3; ++d) e[d] = P[d] - P[3 + d];
    const double c2 = dot3(e, e);
    const double ca = dot3(dir + 3, dir + 6), cb = dot3(dir, dir + 6), cg = dot3(dir, dir + 3);
    const double ra = a2 / b2, rc = c2 / b2;
    // u = s2/s1 = N(v) / (2 D(v));  N^2 - 4 cg N D + 4 Q D^2 = 0   (lowest power first)
    const double N[3] = {rc - ra - 1.0, 2.0 * (ra - rc) * cb, 1.0 - ra + rc};
    const double D[2] = {-cg, ca};
    const double Q[3] = {1.0 - rc, 2.0 * rc * cb, -rc};
    const double DD[3] = {D[0] * D[0], 2.0 * D[0] * D[1], D[1] * D[1]};
    double qc[5] = {0, 0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) qc[i + j] += N[i] * N[j] + 4.0 * Q[i] * DD[j];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j) qc[i + j] -= 4.0 * cg * N[i] * D[j];
    double scale = 0.0;
    bool finite = true;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      scale = fmax(scale, fabs(qc[i]));
      finite = finite && isfinite(qc[i]);
    }
    double vr[4];
    const int nr = (finite && fabs(qc[4]) >= 1e-300) ? quartic_real_roots(qc, vr) : 0;
    double om[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) om[d] = (org[d] + org[3 + d] + org[6 + d]) / 3.0;
    for (int k = 0; k < nr; ++k) {
      const double v = vr[k];
      if (!(v > 0.0) || fabs(poly4(qc, v)) > 1e-6 * scale * fmax(1.0, v * v * v * v)) continue;
      const double den = 2.0 * (D[1] * v + D[0]);
      if (fabs(den) < 1e-12) continue;
      const double u = ((N[2] * v + N[1]) * v + N[0]) / den;
      const double w = 1.0 + v * v - 2.0 * v * cb;
      if (!(u > 0.0) || !(w > 0.0)) continue;
      const double s1 = sqrt(b2 / w);
      double lam[3] = {s1, u * s1, v * s1};
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const double off[3] = {org[3 * i] - om[0], org[3 * i + 1] - om[1], org[3 * i + 2] - om[2]};
        lam[i] -= dot3(dir + 3 * i, off);
      }
      // Newton on g = (|X1-X2|^2 - c2, |X1-X3|^2 - b2, |X2-X3|^2 - a2),  X_i = o_i + lam_i d_i
      double X[9];
      bool good = true;
      for (int it = 0; it <= P3P_NEWTON_ITERS; ++it) {
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int d = 0; d < 3; ++d) X[3 * i + d] = org[3 * i + d] + lam[i] * dir[3 * i + d];
        double e12[3], e13[3], e23[3];
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          e12[d] = X[d] - X[3 + d];
          e13[d] = X[d] - X[6 + d];
          e23[d] = X[3 + d] - X[6 + d];
        }
        const double g0 = dot3(e12, e12) - c2, g1 = dot3(e13, e13) - b2, g2 = dot3(e23, e23) - a2;
        if (it == P3P_NEWTON_ITERS) {
          good = lam[0] > 0.0 && lam[1] > 0.0 && lam[2] > 0.0 &&
                 fmax(fabs(g0), fmax(fabs(g1), fabs(g2))) < 1e-9 * fmax(a2, fmax(b2, c2));
          break;
        }
        // J = 2 [[j00, j01, 0], [j10, 0, j12], [0, j21, j22]]
        const double j00 = 2.0 * dot3(e12, dir), j01 = -2.0 * dot3(e12, dir + 3);
        const double j10 = 2.0 * dot3(e13, dir), j12 = -2.0 * dot3(e13, dir + 6);
        const double j21 = 2.0 * dot3(e23, dir + 3), j22 = -2.0 * dot3(e23, dir + 6);
        const double det = -j00 * j12 * j21 - j01 * j10 * j22;
        if (!isfinite(det) || fabs(det) < 1e-300) {
          good = false;
          break;
        }
        // Cramer
        const double d0 = g0 * (-j12 * j21) - j01 * (g1 * j22 - j12 * g2);
        const double d1 = j00 * (g1 * j22 - j12 * g2) - g0 * (j10 * j22);
        const double d2 = j00 * (-j21 * g1) - j01 * (j10 * g2) + g0 * (j10 * j21);
        lam[0] -= d0 / det;
        lam[1] -= d1 / det;
        lam[2] -= d2 / det;
      }
      if (!good) continue;
      // pose: P_i = R X_i + t
      double Fp[9], Fx[9], M[12];
      triangle_frame(P, Fp);
      triangle_frame(X, Fx);
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) M[4 * i + j] = Fp[i] * Fx[j] + Fp[3 + i] * Fx[3 + j] + Fp[6 + i] * Fx[6 + j];
      double mp[3], mx[3];
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        mp[d] = (P[d] + P[3 + d] + P[6 + d]) / 3.0;
        mx[d] = (X[d] + X[3 + d] + X[6 + d]) / 3.0;
      }
#pragma unroll
      for (int i = 0; i < 3; ++i) M[4 * i + 3] = mp[i] - (M[4 * i] * mx[0] + M[4 * i + 1] * mx[1] + M[4 * i + 2] * mx[2]);
      // bearing residual of the fourth correspondence
      const double dp[3] = {P[9] - M[3], P[10] - M[7], P[11] - M[11]};
      const double* C = rig.Rt[cam4];
      double yb[3], xc[3];
#pragma unroll
      for (int i = 0; i < 3; ++i) yb[i] = M[i] * dp[0] + M[4 + i] * dp[1] + M[8 + i] * dp[2] - C[4 * i + 3];
#pragma unroll
      for (int i = 0; i < 3; ++i) xc[i] = C[i] * yb[0] + C[4 + i] * yb[1] + C[8 + i] * yb[2];
      const double res = 1.0 - dot3(f4, xc) / sqrt(dot3(xc, xc));
      if (res < best_res) {
        best_res = res;
#pragma unroll
        for (int i = 0; i < 12; ++i) best_M[i] = M[i];
      }
    }
    ok = best_res < CUDART_INF;
  }
  HypRec rec;
  if (ok) make_scoring_transforms(best_M, rig, rec, tc_tile, (int)threadIdx.x, tc_mode);
  else make_failed_model(rig, rec, tc_tile, (int)threadIdx.x, tc_mode);
  recs[(size_t)b * n_hyp + h] = rec;
  counts[(size_t)b * n_hyp + h] = ok ? 0 : -(1 << 30);
}

constexpr int RS_THREADS = 128;
constexpr int RS_HPT = 4;                       // hypotheses per thread = 2 packed pairs
constexpr int RS_TILE_H = RS_THREADS * RS_HPT;  // hypotheses per block
constexpr int RS_CHUNK = 512;                   // correspondences per block (64 B each in shared memory)
constexpr int RS_BATCH = 32;                    // correspondences per branch-free batch
constexpr int RS_QCAP = 2048;                   // deferred (batch, hypothesis) re-evaluations per block (expected: a few)

// Blackwell packed FP32: one FFMA2 / FMUL2 / FADD2 instruction does two IEEE float32 operations on a 64-bit register
// pair (SASS FFMA2 / FMUL2 / FADD2, sm_100+).  Each lane rounds exactly like fmaf / fmul / fadd, so the guard-band
// analysis above is unchanged; the point is the halved instruction-issue count (the scalar kernel was issue bound).
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(reinterpret_cast<uint64_t&>(d))
      : "l"(reinterpret_cast<uint64_t&>(a)), "l"(reinterpret_cast<uint64_t&>(b)), "l"(reinterpret_cast<uint64_t&>(c)));
  return d;
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  float2 d;
  asm("mul.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<uint64_t&>(d))
      : "l"(reinterpret_cast<uint64_t&>(a)), "l"(reinterpret_cast<uint64_t&>(b)));
  return d;
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  float2 d;
  asm("add.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<uint64_t&>(d))
      : "l"(reinterpret_cast<uint64_t&>(a)), "l"(reinterpret_cast<uint64_t&>(b)));
  return d;
}
__device__ __forceinline__ float2 fabs2(float2 a) {
  return make_float2(fabsf(a.x), fabsf(a.y));
}
// sign bit of a float as 0 / 1 (1 for negative, -0 and negative NaN)
__device__ __forceinline__ int neg_bit(float v) { return (int)(__float_as_uint(v) >> 31); }

// Shared-memory record of one correspondence: every component duplicated so that one LDS.128 hands the packed
// arithmetic its (v, v) operands without any register shuffling.  q holds p_cur NEGATED (EUCLID) or f_cur (BEARING).
struct __align__(16) PointRec {
  float2 px, py;  // 16 B
  float2 pz, g;   // additive term of t = D - g:  thr^2 - guard_j (EUCLID), -guard_j (BEARING)
  float2 qx, qy;
  float2 qz, pad; // additive term of u = D + g:  thr^2 + guard_j (EUCLID), +guard_j (BEARING)
};

// Decision variable of two hypotheses (packed lanes) for one correspondence: returns t ~ D - g and u ~ D + g.
// certain inlier <=> t > 0, certain outlier <=> u < 0 (i.e. D < -g); anything else is uncertain.
template <int MODE>
__device__ __forceinline__ void decision2(const float2* __restrict__ A, const PointRec& c, const float2 k_a, const float2 k_b,
                                          float2& t, float2& u) {
  const float2 x = ffma2(A[2], c.pz, ffma2(A[1], c.py, ffma2(A[0], c.px, A[9])));
  const float2 y = ffma2(A[5], c.pz, ffma2(A[4], c.py, ffma2(A[3], c.px, A[10])));
  const float2 z = ffma2(A[8], c.pz, ffma2(A[7], c.py, ffma2(A[6], c.px, A[11])));
  if (MODE == SOS_SCORE_EUCLID) {
    const float2 dx = fadd2(x, c.qx), dy = fadd2(y, c.qy), dz = fadd2(z, c.qz);  // q = -p_cur
    const float2 r2 = ffma2(dz, dz, ffma2(dy, dy, fmul2(dx, dx)));
    // D = thr^2 - r2, g = guard_j: the record carries thr^2 - g and thr^2 + g (k_b = -1)
    t = ffma2(r2, k_b, c.g);
    u = ffma2(r2, k_b, c.pad);
  } else {
    const float2 s = ffma2(c.qz, z, ffma2(c.qy, y, fmul2(c.qx, x)));
    const float2 n2 = ffma2(z, z, ffma2(y, y, fmul2(x, x)));
    const float2 sa = fabs2(s);
    // D = s|s| - c^2 n2, g = g_rel n2 + guard_j:  t = s|s| - (c^2 + g_rel) n2 - guard_j,  u = s|s| - (c^2 - g_rel) n2 + guard_j
    // (k_a = -(c^2 + g_rel), k_b = -(c^2 - g_rel); the record carries -guard_j and +guard_j)
    t = ffma2(s, sa, ffma2(n2, k_a, c.g));
    u = ffma2(s, sa, ffma2(n2, k_b, c.pad));
  }
}

// A thread owns RS_HPT hypotheses as RS_HPT/2 packed pairs (24 registers per pair) and walks the block's chunk of
// correspondences in shared memory; every lane reads the SAME correspondence (broadcast LDS.128 x4).  The stacked
// correspondence list is camera-sorted (top view first, pose_est_tools.py:752-778): at most one camera switch per chunk,
// found during staging, so the transforms are loaded once per camera run.  The loop body is branch free: per hypothesis
// two counters, nlo += sign(D - g) and nhi += sign(D + g); nlo == nhi over a batch of RS_BATCH correspondences means no
// pair of the batch was inside the guard band.  Otherwise the (batch, hypothesis) is queued and re-decided after the
// loop, uncertain pairs in float64 — keeping that path out of the loop keeps the warps converged (measured: the
// in-loop version ran with 24 of 32 lanes active).
template <int MODE, int HPT, int CHUNK, int MINB>
__global__ void __launch_bounds__(RS_THREADS, MINB)
score_kernel(const float* __restrict__ p_ref, const float* __restrict__ q_arr, const uint8_t* __restrict__ cam,
             const int32_t* __restrict__ n_arr, int cap, const HypRec* __restrict__ recs, int n_hyp, ScoreConst k,
             const __grid_constant__ Rig rig, int32_t* __restrict__ counts, int32_t* __restrict__ stats) {
  __shared__ PointRec pts[CHUNK];
  __shared__ unsigned char pcam[CHUNK];
  __shared__ float pguard[CHUNK];
  __shared__ uint32_t queue[RS_QCAP];
  __shared__ int queue_n, switch_count, switch_at;
  const int b = blockIdx.z;
  const int n = n_arr[b];
  const int j0 = blockIdx.y * CHUNK;
  if (j0 >= n) return;
  const int nj = min(CHUNK, n - j0);
  const bool multi_cam = rig.n_cams > 1 && cam != nullptr;
  if (threadIdx.x == 0) {
    queue_n = 0;
    switch_count = 0;
    switch_at = 0;
  }
  __syncthreads();
  const float qsign = MODE == SOS_SCORE_EUCLID ? -1.f : 1.f;
  for (int j = threadIdx.x; j < nj; j += RS_THREADS) {
    const size_t o = ((size_t)b * cap + j0 + j) * 3;
    const int c = multi_cam ? (cam[(size_t)b * cap + j0 + j] ? 1 : 0) : 0;
    if (multi_cam && j > 0 && ((cam[(size_t)b * cap + j0 + j - 1] ? 1 : 0) != c)) {
      atomicAdd(&switch_count, 1);
      switch_at = j;  // only read when there is exactly one switch
    }
    const float px = p_ref[o], py = p_ref[o + 1], pz = p_ref[o + 2];
    const float qx = q_arr[o], qy = q_arr[o + 1], qz = q_arr[o + 2];
    const float g = guard_of(MODE, px, py, pz, qx, qy, qz, k.thr);
    PointRec r;
    const float base = MODE == SOS_SCORE_EUCLID ? k.thr_sq : 0.f;
    r.px = make_float2(px, px); r.py = make_float2(py, py); r.pz = make_float2(pz, pz);
    r.g = make_float2(base - g, base - g);
    r.qx = make_float2(qsign * qx, qsign * qx); r.qy = make_float2(qsign * qy, qsign * qy);
    r.qz = make_float2(qsign * qz, qsign * qz);
    r.pad = make_float2(base + g, base + g);
    pts[j] = r;
    pcam[j] = (unsigned char)c;
    pguard[j] = g;
  }
  constexpr int NP = HPT / 2;
  float2 A[NP][12];
  int cnt[HPT];
  const HypRec* rec[HPT];
#pragma unroll
  for (int r = 0; r < HPT; ++r) {
    int h = blockIdx.x * (RS_THREADS * HPT) + r * RS_THREADS + threadIdx.x;
    if (h >= n_hyp) h = n_hyp - 1;  // duplicate work, never stored
    rec[r] = recs + (size_t)b * n_hyp + h;
    cnt[r] = 0;
  }
  const float ka = MODE == SOS_SCORE_EUCLID ? 0.f : -(k.cos_min_sq + k.guard_rel);
  const float kb = MODE == SOS_SCORE_EUCLID ? -1.f : -(k.cos_min_sq - k.guard_rel);
  const float2 k_a = make_float2(ka, ka), k_b = make_float2(kb, kb);
  __syncthreads();
  const int n_switch = switch_count;
  const int split = n_switch == 0 ? nj : (n_switch == 1 ? switch_at : 0);
  // generic camera order (n_switch > 1): every run of equal camera index is handled like a sorted run
  int j_begin = 0;
  while (j_begin < nj) {
    const int c = pcam[j_begin];
    int j_end;
    if (n_switch <= 1) {
      j_end = (j_begin < split) ? split : nj;
    } else {
      j_end = j_begin + 1;
      while (j_end < nj && pcam[j_end] == c) ++j_end;
    }
#pragma unroll
    for (int pr = 0; pr < NP; ++pr)
#pragma unroll
      for (int i = 0; i < 12; ++i)
        A[pr][i] = make_float2(__ldg(&rec[2 * pr]->xf[c][i]), __ldg(&rec[2 * pr + 1]->xf[c][i]));
    for (int jb = j_begin; jb < j_end; jb += RS_BATCH) {
      const int je = min(j_end, jb + RS_BATCH);
      int nlo[HPT], nhi[HPT];
#pragma unroll
      for (int r = 0; r < HPT; ++r) nlo[r] = nhi[r] = 0;
#pragma unroll(HPT == 2 ? 4 : 2)
      for (int j = jb; j < je; ++j) {
        const PointRec pt = pts[j];
#pragma unroll
        for (int pr = 0; pr < NP; ++pr) {
          float2 t, u;
          decision2<MODE>(A[pr], pt, k_a, k_b, t, u);
          nlo[2 * pr] += neg_bit(t.x);
          nlo[2 * pr + 1] += neg_bit(t.y);
          nhi[2 * pr] += neg_bit(u.x);
          nhi[2 * pr + 1] += neg_bit(u.y);
        }
      }
#pragma unroll
      for (int r = 0; r < HPT; ++r) {
        if (nlo[r] == nhi[r]) {
          cnt[r] += (je - jb) - nlo[r];  // all decided: inliers = pairs whose D - g is not negative
        } else {  // rare; two instructions long so that the warp stays converged
          const int slot = atomicAdd(&queue_n, 1);
          if (slot < RS_QCAP) queue[slot] = ((uint32_t)jb << 16) | ((uint32_t)(je - jb) << 10) | ((uint32_t)r << 8) | threadIdx.x;
        }
      }
    }
    j_begin = j_end;
  }
  __syncthreads();
  int nq = queue_n;
  if (stats && threadIdx.x == 0) {   // sos_ransac_score_probe
    atomicAdd(&stats[SOS_STAT_FMA_ENTRIES], nq);
    if (nq > RS_QCAP) atomicAdd(&stats[SOS_STAT_FMA_OVERFLOW_BLOCKS], 1);
  }
  if (nq > RS_QCAP) {  // block-uniform; near-threshold pairs in most batches of most hypotheses: redo the whole chunk in float64
    nq = 0;
#pragma unroll 1
    for (int r = 0; r < HPT; ++r) {
      cnt[r] = 0;
#pragma unroll 1
      for (int j = 0; j < nj; ++j) {
        const PointRec pt = pts[j];
        const float4 p = make_float4(pt.px.x, pt.py.x, pt.pz.x, 0.f);
        const float4 q = make_float4(qsign * pt.qx.x, qsign * pt.qy.x, qsign * pt.qz.x, 0.f);
        cnt[r] += inlier_exact(MODE, rec[r]->pose64, rig, (int)pcam[j], p, q, k.thr) ? 1 : 0;
      }
    }
  }
#pragma unroll
  for (int r = 0; r < HPT; ++r) {
    const int h = blockIdx.x * (RS_THREADS * HPT) + r * RS_THREADS + threadIdx.x;
    if (h < n_hyp && cnt[r] != 0) atomicAdd(&counts[(size_t)b * n_hyp + h], cnt[r]);
  }
  // deferred pass: queue entry = (first point, length <= RS_BATCH, hypothesis slot r, owning thread); every pair of the
  // entry is re-classified with the scalar form of the same arithmetic, uncertain ones by the exact float64 path
  for (int e = threadIdx.x; e < nq; e += RS_THREADS) {
    const uint32_t v = queue[e];
    const int jb = (int)(v >> 16), len = (int)((v >> 10) & 0x3F), r = (int)((v >> 8) & 0x3), t = (int)(v & 0xFF);
    const int h = blockIdx.x * (RS_THREADS * HPT) + r * RS_THREADS + t;
    if (h >= n_hyp) continue;
    const HypRec* hr = recs + (size_t)b * n_hyp + h;
    int add = 0;
    for (int j = jb; j < jb + len; ++j) {
      const PointRec pt = pts[j];
      const float4 p = make_float4(pt.px.x, pt.py.x, pt.pz.x, 0.f);
      const float4 q = make_float4(qsign * pt.qx.x, qsign * pt.qy.x, qsign * pt.qz.x, 0.f);
      const int c = (int)pcam[j];
      float Ax[12];
#pragma unroll
      for (int i = 0; i < 12; ++i) Ax[i] = __ldg(&hr->xf[c][i]);
      float D, g;
      decision<MODE>(Ax, p, q, pguard[j], k, D, g);
      if (fabsf(D) < g) add += inlier_exact(MODE, hr->pose64, rig, c, p, q, k.thr) ? 1 : 0;
      else add += (D > 0.f) ? 1 : 0;
    }
    if (add) atomicAdd(&counts[(size_t)b * n_hyp + h], add);
  }
}

__global__ void __launch_bounds__(1024)
argmax_kernel(const int32_t* __restrict__ counts, const HypRec* __restrict__ recs, int n_hyp, int hyp_offset,
              float* __restrict__ best_pose, int32_t* __restrict__ best_hyp, int32_t* __restrict__ best_count,
              uint64_t* __restrict__ best_key, HypRec* __restrict__ best_rec) {
  __shared__ unsigned long long warp_best[32];
  const int b = blockIdx.x;
  unsigned long long best = 0ull;
  for (int h = threadIdx.x; h < n_hyp; h += blockDim.x) {
    const int c = counts[(size_t)b * n_hyp + h];
    if (c >= 0) {
      const unsigned long long key = ((unsigned long long)(c + 1) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)(hyp_offset + h));
      best = max(best, key);
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) best = max(best, __shfl_xor_sync(0xFFFFFFFFu, best, off));
  if ((threadIdx.x & 31) == 0) warp_best[threadIdx.x >> 5] = best;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) best = max(best, warp_best[w]);
    if (best_key) best_key[b] = best;
    const bool any = best != 0ull;
    const int h = any ? (int)((0xFFFFFFFFu - (uint32_t)(best & 0xFFFFFFFFull)) - (uint32_t)hyp_offset) : -1;
    best_hyp[b] = any ? hyp_offset + h : -1;
    best_count[b] = any ? (int)(best >> 32) - 1 : -1;
    HypRec rec;
    if (any) {
      rec = recs[(size_t)b * n_hyp + h];
    } else {
      for (int i = 0; i < 12; ++i) {
        rec.pose[i] = CUDART_NAN_F;
        rec.pose64[i] = CUDART_NAN;
      }
      for (int c = 0; c < RS_MAX_CAMS; ++c)
        for (int i = 0; i < 12; ++i) rec.xf[c][i] = CUDART_NAN_F;
    }
    best_rec[b] = rec;
    for (int i = 0; i < 12; ++i) best_pose[(size_t)b * 12 + i] = rec.pose[i];
  }
}

// Inlier mask of one hypothesis per problem: evaluated entirely by the exact path (n evaluations, negligible),
// which by construction agrees with every decision the scoring kernel took.
__global__ void __launch_bounds__(256)
mask_kernel(int mode, const float* __restrict__ p_ref, const float* __restrict__ q_arr, const uint8_t* __restrict__ cam,
            const int32_t* __restrict__ n_arr, int cap, const HypRec* __restrict__ best_rec, const __grid_constant__ Rig rig, double thr,
            uint8_t* __restrict__ mask, int32_t* __restrict__ count_out) {
  const int b = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = n_arr[b];
  bool in = false;
  if (j < cap) {
    if (j < n) {
      const size_t o = ((size_t)b * cap + j) * 3;
      const int c = (rig.n_cams > 1 && cam) ? (cam[(size_t)b * cap + j] ? 1 : 0) : 0;
      const float4 p = make_float4(p_ref[o], p_ref[o + 1], p_ref[o + 2], 0.f);
      const float4 q = make_float4(q_arr[o], q_arr[o + 1], q_arr[o + 2], 0.f);
      in = inlier_exact(mode, best_rec[b].pose64, rig, c, p, q, thr);
    }
    if (mask) mask[(size_t)b * cap + j] = in ? 1 : 0;
  }
  if (count_out) {
    const unsigned vote = __ballot_sync(0xFFFFFFFFu, in);
    if ((threadIdx.x & 31) == 0 && vote) atomicAdd(&count_out[b], __popc(vote));
  }
}

// generic k-point Arun, one thread per set (parity with transformations.superimposition_matrix)
__global__ void arun_batch_kernel(const double* __restrict__ v0, const double* __restrict__ v1, int n_sets, int k,
                                  int with_scale, double* __restrict__ M, uint8_t* __restrict__ ok) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_sets) return;
  const double* a = v0 + (size_t)s * k * 3;
  const double* b = v1 + (size_t)s * k * 3;
  double out[12];
  const bool good = arun_fit(a, b, k, out);
  if (good && with_scale) {
    // Umeyama: uniform scale = ratio of the RMS deviations from the centroids (transformations.py:971-975)
    double c0[3] = {0, 0, 0}, c1[3] = {0, 0, 0}, s0 = 0.0, s1 = 0.0;
    for (int i = 0; i < k; ++i)
      for (int d = 0; d < 3; ++d) { c0[d] += a[3 * i + d]; c1[d] += b[3 * i + d]; }
    for (int d = 0; d < 3; ++d) { c0[d] /= (double)k; c1[d] /= (double)k; }
    for (int i = 0; i < k; ++i)
      for (int d = 0; d < 3; ++d) {
        s0 += (a[3 * i + d] - c0[d]) * (a[3 * i + d] - c0[d]);
        s1 += (b[3 * i + d] - c1[d]) * (b[3 * i + d] - c1[d]);
      }
    const double sc = sqrt(s1 / s0);
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) out[r * 4 + c] *= sc;
      out[r * 4 + 3] = c1[r] - (out[r * 4] * c0[0] + out[r * 4 + 1] * c0[1] + out[r * 4 + 2] * c0[2]);
    }
  }
  for (int i = 0; i < 12; ++i) M[(size_t)s * 12 + i] = good ? out[i] : CUDART_NAN;
  if (ok) ok[s] = good ? 1 : 0;
}

// Arun refit over the inlier set: one block per problem, float64 accumulation, two passes (centroids, covariance).
__global__ void __launch_bounds__(1024)
refit_kernel(const float* __restrict__ p_ref, const float* __restrict__ p_cur, const uint8_t* __restrict__ mask,
             const int32_t* __restrict__ n_arr, int cap, float* __restrict__ pose, int32_t* __restrict__ n_used) {
  __shared__ double red[32][16];
  __shared__ double cen[6];
  __shared__ int cnt_sh;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = n_arr[b];
  double acc[16];
  // pass 1: centroids
  for (int i = 0; i < 16; ++i) acc[i] = 0.0;
  for (int j = tid; j < n; j += blockDim.x) {
    if (!mask[(size_t)b * cap + j]) continue;
    const size_t o = ((size_t)b * cap + j) * 3;
    for (int d = 0; d < 3; ++d) { acc[d] += (double)p_cur[o + d]; acc[3 + d] += (double)p_ref[o + d]; }
    acc[6] += 1.0;
  }
  for (int i = 0; i < 7; ++i) {
    double v = acc[i];
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, off);
    if (lane == 0) red[warp][i] = v;
  }
  __syncthreads();
  if (tid == 0) {
    double tot[7];
    for (int i = 0; i < 7; ++i) { tot[i] = 0; for (int w = 0; w < 32; ++w) tot[i] += red[w][i]; }
    cnt_sh = (int)tot[6];
    for (int i = 0; i < 6; ++i) cen[i] = tot[6] > 0 ? tot[i] / tot[6] : 0.0;
  }
  __syncthreads();
  // pass 2: covariance of centred points
  for (int i = 0; i < 16; ++i) acc[i] = 0.0;
  for (int j = tid; j < n; j += blockDim.x) {
    if (!mask[(size_t)b * cap + j]) continue;
    const size_t o = ((size_t)b * cap + j) * 3;
    const double a[3] = {(double)p_cur[o] - cen[0], (double)p_cur[o + 1] - cen[1], (double)p_cur[o + 2] - cen[2]};
    const double c[3] = {(double)p_ref[o] - cen[3], (double)p_ref[o + 1] - cen[4], (double)p_ref[o + 2] - cen[5]};
    for (int r = 0; r < 3; ++r)
      for (int s = 0; s < 3; ++s) acc[r * 3 + s] += c[r] * a[s];
  }
  __syncthreads();
  for (int i = 0; i < 9; ++i) {
    double v = acc[i];
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, off);
    if (lane == 0) red[warp][i] = v;
  }
  __syncthreads();
  if (tid == 0) {
    double Hm[9], R[9];
    for (int i = 0; i < 9; ++i) { Hm[i] = 0; for (int w = 0; w < 32; ++w) Hm[i] += red[w][i]; }
    const bool ok = cnt_sh >= 3 && kabsch_rotation(Hm, R);
    if (n_used) n_used[b] = ok ? cnt_sh : -1;
    for (int r = 0; r < 3; ++r) {
      for (int s = 0; s < 3; ++s) pose[(size_t)b * 12 + r * 4 + s] = ok ? (float)R[r * 3 + s] : CUDART_NAN_F;
      pose[(size_t)b * 12 + r * 4 + 3] =
          ok ? (float)(cen[3 + r] - (R[r * 3] * cen[0] + R[r * 3 + 1] * cen[1] + R[r * 3 + 2] * cen[2])) : CUDART_NAN_F;
    }
  }
}

int fill_rig(const double* rig, int n_cams, Rig& out) {
  out.n_cams = n_cams < 1 ? 1 : n_cams;
  for (int c = 0; c < RS_MAX_CAMS; ++c)
    for (int i = 0; i < 12; ++i) out.Rt[c][i] = (i == 0 || i == 5 || i == 10) ? 1.0 : 0.0;
  if (rig)
    for (int c = 0; c < n_cams; ++c)
      for (int i = 0; i < 12; ++i) out.Rt[c][i] = rig[c * 12 + i];
  return 0;
}

ScoreConst make_const(int mode, double thr) {
  ScoreConst k;
  k.thr_sq = (float)(thr * thr);
  k.cos_min_sq = (float)((1.0 - thr) * (1.0 - thr));
  k.guard_rel = (float)(80.0 * 5.9604644775390625e-08 * 1.0001);
  k.thr = thr;
  (void)mode;
  return k;
}

struct RansacScratch {
  HypRec* recs;
  int32_t* counts;
  HypRec* best_rec;
  uint8_t *tc_a, *tc_b;          // tensor-core score engine: hypothesis tiles, correspondence tiles (score_mma.cuh)
  score_tc::TileMeta* tc_meta;
};

int ransac_scratch(sos_ctx* ctx, int n_problems, int n_hyp, int tc_cap, RansacScratch& s) {
  const size_t rec_bytes = sos_align_up((size_t)n_problems * n_hyp * sizeof(HypRec), 256);
  const size_t cnt_bytes = sos_align_up((size_t)n_problems * n_hyp * sizeof(int32_t), 256);
  const size_t best_bytes = sos_align_up((size_t)n_problems * sizeof(HypRec), 256);
  const size_t ht = (size_t)sos_div_up(n_hyp, score_tc::TILE), ct = (size_t)sos_div_up(tc_cap > 0 ? tc_cap : 1, score_tc::TILE);
  const size_t a_bytes = tc_cap > 0 ? (size_t)n_problems * ht * 2 * score_tc::TILE_BYTES : 0;
  const size_t b_bytes = tc_cap > 0 ? (size_t)n_problems * ct * 2 * score_tc::TILE_BYTES : 0;
  const size_t m_bytes = tc_cap > 0 ? sos_align_up((size_t)n_problems * ct * sizeof(score_tc::TileMeta), 256) : 0;
  void* base = nullptr;
  const int rc = sos_arena_get(ctx, rec_bytes + cnt_bytes + best_bytes + a_bytes + b_bytes + m_bytes + 1024, &base);
  if (rc != SOS_OK) return rc;
  char* p = (char*)base;
  s.recs = (HypRec*)p; p += rec_bytes;
  s.counts = (int32_t*)p; p += cnt_bytes;
  s.best_rec = (HypRec*)p; p += best_bytes;
  p = (char*)sos_align_up((size_t)(uintptr_t)p, 1024);
  s.tc_a = tc_cap > 0 ? (uint8_t*)p : nullptr; p += a_bytes;
  s.tc_b = tc_cap > 0 ? (uint8_t*)p : nullptr; p += b_bytes;
  s.tc_meta = tc_cap > 0 ? (score_tc::TileMeta*)p : nullptr;
  return SOS_OK;
}

// Both scores on the tensor cores (score_mma.cuh).  SOS_SCORE_ENGINE=fma keeps the FP32-pipe kernel; tests/test_gpu_ransac.py
// runs every case on both.
bool use_tensor_score(int score_mode, int n_hyp, int cap) {
  (void)score_mode;   // both scores have a tensor-core engine
  if (n_hyp < 32 || cap < 1) return false;
  const char* e = getenv("SOS_SCORE_ENGINE");
  return !(e && e[0] == 'f');
}

int launch_score_tc(sos_ctx* ctx, int mode, const Rig& rig, const RansacScratch& s, const float* p_ref, const float* f_cur, const uint8_t* cam,
                    const int32_t* n, int n_problems, int cap, int n_hyp, ScoreConst k, float* probe, int32_t* stats) {
  using namespace score_tc;
  const int ht = sos_div_up(n_hyp, TILE), ct = sos_div_up(cap, TILE);
  corr_expand_kernel<<<dim3(ct, n_problems), TILE, 0, ctx->stream>>>(mode, p_ref, f_cur, cam, n, cap, rig.n_cams, ct, s.tc_b, s.tc_meta);
  SOS_LAUNCHED_AS(ctx, "score_expand_kernel");
  Args a;
  a.a_exp = s.tc_a; a.b_exp = s.tc_b; a.meta = s.tc_meta; a.n_arr = n;
  a.cap = cap; a.n_hyp = n_hyp; a.ht = ht; a.ct = ct;
  // work items = problems x hypothesis tiles x splits of the correspondence range: at least two per SM, a few tiles per item
  // at least, and among the candidates the split with the smallest loss to the last, partly filled wave of CTAs (one CTA
  // per SM at a time: 512 items on 148 SMs would idle 13 % of the machine, 1024 items 1 %)
  const int max_splits = sos_div_up(ct, 4);
  int splits = sos_div_up(2 * ctx->sm_count, n_problems * ht);
  splits = splits < 1 ? 1 : (splits > max_splits ? max_splits : splits);
  {
    double best_loss = 1e30;
    int best = splits;
    for (int sp = splits; sp <= max_splits && sp < splits + 8; ++sp) {
      const long long items = (long long)n_problems * ht * sp;
      const long long waves = (items + ctx->sm_count - 1) / ctx->sm_count;
      const double loss = (double)(waves * ctx->sm_count) / (double)items * (1.0 + 0.01 * (sp - splits));   // (a split costs a prologue)
      if (loss < best_loss - 1e-9) { best_loss = loss; best = sp; }
    }
    splits = best;
  }
  a.splits = splits;
  a.recs = s.recs; a.counts = s.counts; a.p_ref = p_ref; a.f_cur = f_cur; a.cam = cam; a.k = k; a.probe = probe; a.stats = stats;
  static bool attr_set[64][4] = {};     // per device: the opt-in to > 48 KB of dynamic shared memory
  const bool euclid = mode == SOS_SCORE_EUCLID;
  const bool diag = probe || stats;
  const int dev = ctx->device & 63, v = (diag ? 1 : 0) + (euclid ? 2 : 0);
  auto kern = diag ? (euclid ? score_mma_kernel<true, SOS_SCORE_EUCLID> : score_mma_kernel<true, SOS_SCORE_BEARING>)
                    : (euclid ? score_mma_kernel<false, SOS_SCORE_EUCLID> : score_mma_kernel<false, SOS_SCORE_BEARING>);
  if (!attr_set[dev][v]) {
    SOS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    attr_set[dev][v] = true;
  }
  const unsigned grid = (unsigned)n_problems * ht * splits;
  kern<<<grid, THREADS, SMEM_BYTES, ctx->stream>>>(a, rig);
  SOS_LAUNCHED_AS(ctx, "score_mma_kernel");
  return SOS_OK;
}

template <int MODE>
int launch_score(sos_ctx* ctx, const Rig& rig, dim3 grid, const float* p_ref, const float* q, const uint8_t* cam,
                 const int32_t* n, int cap, const HypRec* recs, int n_hyp, ScoreConst k, int32_t* counts, int32_t* stats) {
  // 4 hypotheses per thread, 512 correspondences per block, 4 blocks per SM.  Measured against higher-occupancy shapes in
  // round 2 (profiles/r02/score_variants_and_ring_depth_ab.log: 2 hypotheses per thread with 6-8 blocks per SM, 256-point
  // chunks): all slower (0.74 - 0.81 ms against 0.72 ms) — fewer hypotheses per shared-memory read and more block prologues
  // cost more than the extra warps hide.
  score_kernel<MODE, RS_HPT, RS_CHUNK, 4><<<grid, RS_THREADS, 0, ctx->stream>>>(p_ref, q, cam, n, cap, recs, n_hyp, k, rig, counts, stats);
  SOS_LAUNCHED_AS(ctx, "score_kernel");
  return SOS_OK;
}

}  // namespace

extern "C" int sos_arun_batch(sos_ctx* ctx, const double* v0, const double* v1, int n_sets, int k, int with_scale,
                              double* M, uint8_t* ok) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n_sets >= 0 && k >= 3, "need k >= 3 points per set");
  if (n_sets == 0) return SOS_OK;
  SOS_CHECK_ARG(v0 && v1 && M, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  arun_batch_kernel<<<sos_div_up(n_sets, 128), 128, 0, ctx->stream>>>(v0, v1, n_sets, k, with_scale, M, ok);
  SOS_LAUNCHED_AS(ctx, "arun_batch_kernel");
  return SOS_OK;
}

namespace {
// solver 0: 3D-3D Arun hypotheses (3 sample numbers per hypothesis); solver 1: bearing-only three-point hypotheses (4 numbers)
int ransac_run(sos_ctx* ctx, int solver, const float* p_ref, const float* p_cur, const float* f_cur,
                              const uint8_t* cam, const int32_t* n, int n_problems, int cap, const double* rig,
                              int n_cams, const uint32_t* hyp, int n_hyp, int hyp_offset, int score_mode,
                              double threshold, float* best_pose, int32_t* best_hyp, int32_t* best_count,
                              uint8_t* inlier_mask, uint64_t* best_key, int32_t* all_counts, float* tc_probe = nullptr,
                              int32_t* stats = nullptr) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n_problems >= 0 && cap >= 0 && n_hyp >= 0, "negative size");
  SOS_CHECK_ARG(score_mode == SOS_SCORE_EUCLID || score_mode == SOS_SCORE_BEARING, "unknown score mode");
  SOS_CHECK_ARG(n_cams >= 0 && n_cams <= RS_MAX_CAMS, "at most 2 cameras in the rig");
  SOS_CHECK_ARG(n_problems <= 65535, "at most 65535 problems per call");
  if (n_problems == 0) return SOS_OK;
  SOS_CHECK_ARG(p_ref && (p_cur || solver == 1) && n && best_pose && best_hyp && best_count, "NULL array");
  SOS_CHECK_ARG(n_hyp == 0 || hyp, "hyp is NULL");
  SOS_CHECK_ARG(score_mode != SOS_SCORE_BEARING || f_cur, "bearing score needs f_cur");
  SOS_CHECK_ARG(score_mode != SOS_SCORE_BEARING || (threshold > 0.0 && threshold < 1.0), "bearing threshold must be in (0,1)");
  SOS_CUDA(cudaSetDevice(ctx->device));
  Rig r;
  fill_rig(score_mode == SOS_SCORE_BEARING ? rig : nullptr, score_mode == SOS_SCORE_BEARING ? n_cams : 1, r);
  const ScoreConst k = make_const(score_mode, threshold);
  RansacScratch s;
  const int n_hyp_alloc = n_hyp > 0 ? n_hyp : 1;
  const bool tc = tc_probe != nullptr || use_tensor_score(score_mode, n_hyp, cap);
  if (stats) SOS_CUDA(cudaMemsetAsync(stats, 0, SOS_SCORE_STATS * sizeof(int32_t), ctx->stream));
  int rc = ransac_scratch(ctx, n_problems, n_hyp_alloc, tc ? cap : 0, s);
  if (rc != SOS_OK) return rc;
  if (n_hyp > 0) {
    dim3 hgrid(sos_div_up(n_hyp, 128), n_problems);
    if (solver == 1)
      hypothesize_p3p_kernel<<<hgrid, 128, 0, ctx->stream>>>(p_ref, f_cur, cam, n, cap, hyp, 0, n_hyp, r, s.recs, s.counts, s.tc_a, score_mode);
    else
      hypothesize_kernel<<<hgrid, 128, 0, ctx->stream>>>(p_ref, p_cur, n, cap, hyp, 0, n_hyp, r, s.recs, s.counts, s.tc_a, score_mode);
    SOS_LAUNCHED_AS(ctx, "hypothesize_kernel");
    if (cap > 0 && tc) {
      rc = launch_score_tc(ctx, score_mode, r, s, p_ref, score_mode == SOS_SCORE_EUCLID ? p_cur : f_cur, cam, n, n_problems, cap, n_hyp, k,
                           tc_probe, stats);
      if (rc != SOS_OK) return rc;
    } else if (cap > 0) {
      dim3 sgrid(sos_div_up(n_hyp, RS_TILE_H), sos_div_up(cap, RS_CHUNK), n_problems);
      const float* q = score_mode == SOS_SCORE_EUCLID ? p_cur : f_cur;
      rc = score_mode == SOS_SCORE_EUCLID
               ? launch_score<SOS_SCORE_EUCLID>(ctx, r, sgrid, p_ref, q, cam, n, cap, s.recs, n_hyp, k, s.counts, stats)
               : launch_score<SOS_SCORE_BEARING>(ctx, r, sgrid, p_ref, q, cam, n, cap, s.recs, n_hyp, k, s.counts, stats);
      if (rc != SOS_OK) return rc;
    }
  }
  argmax_kernel<<<n_problems, n_hyp > 8192 ? 1024 : 256, 0, ctx->stream>>>(s.counts, s.recs, n_hyp, hyp_offset, best_pose, best_hyp,
                                                     best_count, best_key, s.best_rec);
  SOS_LAUNCHED_AS(ctx, "argmax_kernel");
  if (all_counts && n_hyp > 0)
    SOS_CUDA(cudaMemcpyAsync(all_counts, s.counts, (size_t)n_problems * n_hyp * sizeof(int32_t), cudaMemcpyDeviceToDevice,
                             ctx->stream));
  if (inlier_mask && cap > 0) {
    dim3 mgrid(sos_div_up(cap, 256), n_problems);
    const float* q = score_mode == SOS_SCORE_EUCLID ? p_cur : f_cur;
    mask_kernel<<<mgrid, 256, 0, ctx->stream>>>(score_mode, p_ref, q, cam, n, cap, s.best_rec, r, threshold, inlier_mask, nullptr);
    SOS_LAUNCHED_AS(ctx, "mask_kernel");
  }
  return SOS_OK;
}
}  // namespace

extern "C" int sos_ransac_p3d(sos_ctx* ctx, const float* p_ref, const float* p_cur, const float* f_cur,
                              const uint8_t* cam, const int32_t* n, int n_problems, int cap, const double* rig,
                              int n_cams, const uint32_t* hyp, int n_hyp, int hyp_offset, int score_mode,
                              double threshold, float* best_pose, int32_t* best_hyp, int32_t* best_count,
                              uint8_t* inlier_mask, uint64_t* best_key, int32_t* all_counts) {
  return ransac_run(ctx, 0, p_ref, p_cur, f_cur, cam, n, n_problems, cap, rig, n_cams, hyp, n_hyp, hyp_offset, score_mode,
                    threshold, best_pose, best_hyp, best_count, inlier_mask, best_key, all_counts);
}

extern "C" int sos_ransac_score_probe(sos_ctx* ctx, const float* p_ref, const float* p_cur, const float* f_cur,
                                      const uint8_t* cam, const int32_t* n, int n_problems, int cap, const double* rig,
                                      int n_cams, const uint32_t* hyp, int n_hyp, int score_mode, double threshold,
                                      float* best_pose, int32_t* best_hyp, int32_t* best_count, int32_t* all_counts,
                                      float* sn, int32_t* stats) {
  SOS_CHECK_ARG(sn || stats, "sn and stats are both NULL");
  return ransac_run(ctx, 0, p_ref, p_cur, f_cur, cam, n, n_problems, cap, rig, n_cams, hyp, n_hyp, 0, score_mode,
                    threshold, best_pose, best_hyp, best_count, nullptr, nullptr, all_counts, sn, stats);
}

extern "C" int sos_ransac_p3p(sos_ctx* ctx, const float* p_ref, const float* f_cur, const uint8_t* cam, const int32_t* n,
                              int n_problems, int cap, const double* rig, int n_cams, const uint32_t* hyp, int n_hyp,
                              int hyp_offset, double threshold, float* best_pose, int32_t* best_hyp, int32_t* best_count,
                              uint8_t* inlier_mask, uint64_t* best_key, int32_t* all_counts) {
  SOS_CHECK_ARG(f_cur || n_problems == 0, "f_cur is NULL");
  return ransac_run(ctx, 1, p_ref, nullptr, f_cur, cam, n, n_problems, cap, rig, n_cams, hyp, n_hyp, hyp_offset,
                    SOS_SCORE_BEARING, threshold, best_pose, best_hyp, best_count, inlier_mask, best_key, all_counts);
}

extern "C" int sos_ransac_p3d_eval(sos_ctx* ctx, const float* p_ref, const float* p_cur, const float* f_cur,
                                   const uint8_t* cam, const int32_t* n, int n_problems, int cap, const double* rig,
                                   int n_cams, const uint32_t* hyp_row, int score_mode, double threshold, float* pose,
                                   int32_t* count, uint8_t* inlier_mask) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n_problems >= 0 && cap >= 0, "negative size");
  SOS_CHECK_ARG(score_mode == SOS_SCORE_EUCLID || score_mode == SOS_SCORE_BEARING, "unknown score mode");
  SOS_CHECK_ARG(n_cams >= 0 && n_cams <= RS_MAX_CAMS, "at most 2 cameras in the rig");
  SOS_CHECK_ARG(n_problems <= 65535, "at most 65535 problems per call");
  if (n_problems == 0) return SOS_OK;
  SOS_CHECK_ARG(p_ref && p_cur && n && hyp_row && pose && count, "NULL array");
  SOS_CHECK_ARG(score_mode != SOS_SCORE_BEARING || f_cur, "bearing score needs f_cur");
  SOS_CUDA(cudaSetDevice(ctx->device));
  Rig r;
  fill_rig(score_mode == SOS_SCORE_BEARING ? rig : nullptr, score_mode == SOS_SCORE_BEARING ? n_cams : 1, r);
  const ScoreConst k = make_const(score_mode, threshold);
  RansacScratch s;
  int rc = ransac_scratch(ctx, n_problems, 1, 0, s);
  if (rc != SOS_OK) return rc;
  dim3 hgrid(1, n_problems);
  // one hypothesis per problem, each with its own row of sample numbers (stride 3 per problem)
  hypothesize_kernel<<<hgrid, 128, 0, ctx->stream>>>(p_ref, p_cur, n, cap, hyp_row, 3, 1, r, s.recs, s.counts, nullptr, score_mode);
  SOS_LAUNCHED_AS(ctx, "hypothesize_kernel");
  // counts[b] is 0 for a valid model and hugely negative otherwise: the mask kernel adds the inliers on top
  SOS_CUDA(cudaMemcpyAsync(count, s.counts, (size_t)n_problems * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
  SOS_CUDA(cudaMemcpy2DAsync(pose, 12 * sizeof(float), (const char*)s.recs + offsetof(HypRec, pose), sizeof(HypRec), 12 * sizeof(float), n_problems,
                             cudaMemcpyDeviceToDevice, ctx->stream));
  if (cap > 0) {
    dim3 mgrid(sos_div_up(cap, 256), n_problems);
    const float* q = score_mode == SOS_SCORE_EUCLID ? p_cur : f_cur;
    mask_kernel<<<mgrid, 256, 0, ctx->stream>>>(score_mode, p_ref, q, cam, n, cap, s.recs, r, threshold, inlier_mask, count);
    SOS_LAUNCHED_AS(ctx, "mask_kernel");
  }
  return SOS_OK;
}

extern "C" int sos_refit_inliers(sos_ctx* ctx, const float* p_ref, const float* p_cur, const uint8_t* inlier_mask,
                                 const int32_t* n, int n_problems, int cap, float* pose, int32_t* n_used) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n_problems >= 0 && cap >= 0, "negative size");
  if (n_problems == 0) return SOS_OK;
  SOS_CHECK_ARG(p_ref && p_cur && inlier_mask && n && pose, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  refit_kernel<<<n_problems, 1024, 0, ctx->stream>>>(p_ref, p_cur, inlier_mask, n, cap, pose, n_used);
  SOS_LAUNCHED_AS(ctx, "refit_kernel");
  return SOS_OK;
}
